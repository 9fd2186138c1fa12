// HBM-bound kernels of the NST evaluation: weight packing, the 3-channel first layer (K0+K1 head,
// and its dgrad tail), 2x2 max-pool fwd/bwd (K2), Gram finalize + loss (K4/K6), content MSE (K6),
// mean/std style statistics (K6, StyleLoss_BN and Classifier2 features).  All NHWC bf16 with
// 128-bit accesses (8 channels per thread), fp32 math, double accumulation of scalar losses.
#include <algorithm>

#include "isx_common.cuh"
#include "isx_internal.h"
#include "isx_kernels.h"

namespace isx {

__constant__ float c_mean[3] = {0.485f, 0.456f, 0.406f};  // models/vgg/vgg.py:66
__constant__ float c_std[3] = {0.229f, 0.224f, 0.225f};

// ------------------------------------------------------------------------------------------
// weight packing: fp32 OIHW -> bf16 [tap][Cout][Cin] (fwd) and [8-tap][Cin][Cout] (dgrad)
// ------------------------------------------------------------------------------------------
__global__ void pack_w_kernel(const float* __restrict__ w, int Cout, int Cin, __nv_bfloat16* __restrict__ wf,
                              __nv_bfloat16* __restrict__ wd) {
  const long n = static_cast<long>(Cout) * Cin * 9;
  for (long i = blockIdx.x * static_cast<long>(blockDim.x) + threadIdx.x; i < n;
       i += static_cast<long>(gridDim.x) * blockDim.x) {
    const int tap = i % 9;
    const int ci = (i / 9) % Cin;
    const int co = i / (9L * Cin);
    const __nv_bfloat16 v = __float2bfloat16_rn(w[i]);
    if (wf) wf[(static_cast<long>(tap) * Cout + co) * Cin + ci] = v;
    if (wd) wd[(static_cast<long>(8 - tap) * Cin + ci) * Cout + co] = v;
  }
}

int pack_conv_weights(const float* w, int Cout, int Cin, __nv_bfloat16* wf, __nv_bfloat16* wd, cudaStream_t s) {
  const long n = static_cast<long>(Cout) * Cin * 9;
  const int blocks = static_cast<int>(std::min<long>((n + 255) / 256, isx_num_sms() * 8));
  pack_w_kernel<<<blocks, 256, 0, s>>>(w, Cout, Cin, wf, wd);
  ISX_LAUNCH_CHECK();
  return 0;
}

// conv1_1 dgrad weights for the tensor-core tail: fp32 [64,3,3,3] -> bf16 [8-tap][16][64], rows 3..15 zero
__global__ void pack_w0_dgrad_kernel(const float* __restrict__ w, __nv_bfloat16* __restrict__ wd) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;  // over 9*16*64
  if (i >= 9 * 16 * 64) return;
  const int o = i % 64, c = (i / 64) % 16, tapd = i / (64 * 16);
  const int tap = 8 - tapd;
  wd[i] = c < 3 ? __float2bfloat16_rn(w[(o * 3 + c) * 9 + tap]) : __float2bfloat16_rn(0.f);
}

int pack_w0_dgrad(const float* w, __nv_bfloat16* wd, cudaStream_t s) {
  pack_w0_dgrad_kernel<<<(9 * 16 * 64 + 255) / 256, 256, 0, s>>>(w, wd);
  ISX_LAUNCH_CHECK();
  return 0;
}

// ------------------------------------------------------------------------------------------
// conv1_1 forward: fp32 NCHW image -> Normalize (-> * mask) -> 3x3 conv (3->64) + bias + ReLU -> bf16 NHWC
// (models/vgg/vgg.py:81-87; K0 fused into K1's first layer)
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128)
conv1_1_fwd_kernel(const float* __restrict__ x, int xc, const float* __restrict__ mask, int mask_b,
                   const float* __restrict__ w, const float* __restrict__ bias, __nv_bfloat16* __restrict__ out, int B,
                   int H, int W) {
  __shared__ float sw[27][64];
  __shared__ float sb[64];
  for (int i = threadIdx.x; i < 27 * 64; i += blockDim.x) {
    const int o = i % 64, k = i / 64;  // k = c*9 + tap in OIHW order
    sw[k][o] = w[o * 27 + k];
  }
  if (threadIdx.x < 64) sb[threadIdx.x] = bias ? bias[threadIdx.x] : 0.f;
  __syncthreads();
  const long npix = static_cast<long>(B) * H * W;
  const long pix = blockIdx.x * static_cast<long>(blockDim.x) + threadIdx.x;
  if (pix >= npix) return;
  const int xx = pix % W;
  const int yy = (pix / W) % H;
  const int b = pix / (static_cast<long>(W) * H);
  float in[27];
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    const float* xp = x + (static_cast<long>(b) * xc + (xc == 3 ? c : 0)) * H * W;
#pragma unroll
    for (int ky = 0; ky < 3; ++ky) {
#pragma unroll
      for (int kx = 0; kx < 3; ++kx) {
        const int y = yy + ky - 1, xq = xx + kx - 1;
        float v = 0.f;
        if (y >= 0 && y < H && xq >= 0 && xq < W) {
          v = (xp[static_cast<long>(y) * W + xq] - c_mean[c]) / c_std[c];
          if (mask) v *= mask[(static_cast<long>(mask_b > 1 ? b : 0) * H + y) * W + xq];
        }
        in[c * 9 + ky * 3 + kx] = v;
      }
    }
  }
  uint4* op = reinterpret_cast<uint4*>(out + pix * 64);
#pragma unroll 1
  for (int g = 0; g < 8; ++g) {
    float acc[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[j] = sb[g * 8 + j];
#pragma unroll
    for (int k = 0; k < 27; ++k) {
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[j] = fmaf(in[k], sw[k][g * 8 + j], acc[j]);
    }
    uint4 o;
    o.x = pack_bf16x2(fmaxf(acc[0], 0.f), fmaxf(acc[1], 0.f));
    o.y = pack_bf16x2(fmaxf(acc[2], 0.f), fmaxf(acc[3], 0.f));
    o.z = pack_bf16x2(fmaxf(acc[4], 0.f), fmaxf(acc[5], 0.f));
    o.w = pack_bf16x2(fmaxf(acc[6], 0.f), fmaxf(acc[7], 0.f));
    op[g] = o;
  }
}

int conv1_1_fwd(const float* x, int xc, const float* mask, int mask_b, const float* w, const float* bias,
                __nv_bfloat16* out, int B, int H, int W, cudaStream_t s) {
  ISX_REQUIRE(xc == 1 || xc == 3, "conv1_1: image must have 1 or 3 channels, got %d", xc);
  const long npix = static_cast<long>(B) * H * W;
  conv1_1_fwd_kernel<<<static_cast<unsigned>((npix + 127) / 128), 128, 0, s>>>(x, xc, mask, mask_b, w, bias, out, B, H, W);
  ISX_LAUNCH_CHECK();
  return 0;
}

// conv1_1 dgrad + Normalize backward: dY bf16 NHWC (64 ch, already ReLU-masked) -> dX fp32 NCHW [B,3,H,W]
__global__ void __launch_bounds__(128)
conv1_1_dgrad_kernel(const __nv_bfloat16* __restrict__ dy, const float* __restrict__ w, const float* __restrict__ mask,
                     int mask_b, float* __restrict__ dx, int xc, int B, int H, int W) {
  __shared__ float sw[9][64][3];  // [tap][o][c]
  for (int i = threadIdx.x; i < 27 * 64; i += blockDim.x) {
    const int tap = i % 9, c = (i / 9) % 3, o = i / 27;
    sw[tap][o][c] = w[i];
  }
  __syncthreads();
  const long npix = static_cast<long>(B) * H * W;
  const long pix = blockIdx.x * static_cast<long>(blockDim.x) + threadIdx.x;
  if (pix >= npix) return;
  const int xx = pix % W;
  const int yy = (pix / W) % H;
  const int b = pix / (static_cast<long>(W) * H);
  float a0 = 0.f, a1 = 0.f, a2 = 0.f;
#pragma unroll 1
  for (int ky = 0; ky < 3; ++ky) {
#pragma unroll 1
    for (int kx = 0; kx < 3; ++kx) {
      // y_out = y_in - (ky - 1): output pixel (yo, xo) used input (yy, xx) with tap (ky, kx)
      const int yo = yy - ky + 1, xo = xx - kx + 1;
      if (yo < 0 || yo >= H || xo < 0 || xo >= W) continue;
      const uint4* p = reinterpret_cast<const uint4*>(dy + ((static_cast<long>(b) * H + yo) * W + xo) * 64);
      const int tap = ky * 3 + kx;
#pragma unroll
      for (int g = 0; g < 8; ++g) {
        const uint4 u = __ldg(p + g);
        const uint32_t uu[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float2 t = unpack_bf16x2(uu[j]);
          const int o = g * 8 + j * 2;
          a0 = fmaf(t.x, sw[tap][o][0], a0); a1 = fmaf(t.x, sw[tap][o][1], a1); a2 = fmaf(t.x, sw[tap][o][2], a2);
          a0 = fmaf(t.y, sw[tap][o + 1][0], a0); a1 = fmaf(t.y, sw[tap][o + 1][1], a1); a2 = fmaf(t.y, sw[tap][o + 1][2], a2);
        }
      }
    }
  }
  float m = 1.f;
  if (mask) m = mask[(static_cast<long>(mask_b > 1 ? b : 0) * H + yy) * W + xx];
  a0 = a0 * m / c_std[0]; a1 = a1 * m / c_std[1]; a2 = a2 * m / c_std[2];
  const long hw = static_cast<long>(H) * W;
  const long off = static_cast<long>(yy) * W + xx;
  if (xc == 3) {
    float* o = dx + static_cast<long>(b) * 3 * hw + off;
    o[0] = a0; o[hw] = a1; o[2 * hw] = a2;
  } else {
    dx[static_cast<long>(b) * hw + off] = a0 + a1 + a2;  // 1-channel image broadcast to 3 (SURVEY note N3)
  }
}

int conv1_1_dgrad(const __nv_bfloat16* dy, const float* w, const float* mask, int mask_b, float* dx, int xc, int B,
                  int H, int W, cudaStream_t s) {
  const long npix = static_cast<long>(B) * H * W;
  conv1_1_dgrad_kernel<<<static_cast<unsigned>((npix + 127) / 128), 128, 0, s>>>(dy, w, mask, mask_b, dx, xc, B, H, W);
  ISX_LAUNCH_CHECK();
  return 0;
}

// ------------------------------------------------------------------------------------------
// 2x2 stride-2 max-pool (torchvision vgg19.features MaxPool2d(2,2)); first maximum in scan order
// wins ties, like ATen's `val > maxval` loop.
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ void unpack8(const uint4& u, float (&f)[8]) {
  float2 t;
  t = unpack_bf16x2(u.x); f[0] = t.x; f[1] = t.y;
  t = unpack_bf16x2(u.y); f[2] = t.x; f[3] = t.y;
  t = unpack_bf16x2(u.z); f[4] = t.x; f[5] = t.y;
  t = unpack_bf16x2(u.w); f[6] = t.x; f[7] = t.y;
}
__device__ __forceinline__ uint4 pack8(const float (&f)[8]) {
  uint4 o;
  o.x = pack_bf16x2(f[0], f[1]); o.y = pack_bf16x2(f[2], f[3]);
  o.z = pack_bf16x2(f[4], f[5]); o.w = pack_bf16x2(f[6], f[7]);
  return o;
}

__global__ void maxpool_fwd_kernel(const __nv_bfloat16* __restrict__ in, __nv_bfloat16* __restrict__ out, int B, int H,
                                   int W, int C) {
  const int Ho = H / 2, Wo = W / 2, C8 = C / 8;
  const long n = static_cast<long>(B) * Ho * Wo * C8;
  for (long i = blockIdx.x * static_cast<long>(blockDim.x) + threadIdx.x; i < n;
       i += static_cast<long>(gridDim.x) * blockDim.x) {
    const int c8 = i % C8;
    const int xo = (i / C8) % Wo;
    const int yo = (i / (static_cast<long>(C8) * Wo)) % Ho;
    const int b = i / (static_cast<long>(C8) * Wo * Ho);
    const __nv_bfloat16* p = in + ((static_cast<long>(b) * H + 2 * yo) * W + 2 * xo) * C + c8 * 8;
    float a[8], t[8];
    unpack8(__ldg(reinterpret_cast<const uint4*>(p)), a);
    unpack8(__ldg(reinterpret_cast<const uint4*>(p + C)), t);
#pragma unroll
    for (int j = 0; j < 8; ++j) a[j] = t[j] > a[j] ? t[j] : a[j];
    unpack8(__ldg(reinterpret_cast<const uint4*>(p + static_cast<long>(W) * C)), t);
#pragma unroll
    for (int j = 0; j < 8; ++j) a[j] = t[j] > a[j] ? t[j] : a[j];
    unpack8(__ldg(reinterpret_cast<const uint4*>(p + static_cast<long>(W) * C + C)), t);
#pragma unroll
    for (int j = 0; j < 8; ++j) a[j] = t[j] > a[j] ? t[j] : a[j];
    *reinterpret_cast<uint4*>(out + ((static_cast<long>(b) * Ho + yo) * Wo + xo) * C + c8 * 8) = pack8(a);
  }
}

int maxpool_fwd(const __nv_bfloat16* in, __nv_bfloat16* out, int B, int H, int W, int C, cudaStream_t s) {
  ISX_REQUIRE(C % 8 == 0 && H >= 2 && W >= 2, "maxpool: bad shape H=%d W=%d C=%d", H, W, C);
  const long n = static_cast<long>(B) * (H / 2) * (W / 2) * (C / 8);
  const int blocks = static_cast<int>(std::min<long>((n + 255) / 256, static_cast<long>(isx_num_sms()) * 16));
  maxpool_fwd_kernel<<<blocks, 256, 0, s>>>(in, out, B, H, W, C);
  ISX_LAUNCH_CHECK();
  return 0;
}

// dx[pre-pool] = (argmax of its window && act > 0) ? dy[pooled] : 0   (max-pool bwd fused with ReLU bwd)
__global__ void maxpool_bwd_kernel(const __nv_bfloat16* __restrict__ dy, const __nv_bfloat16* __restrict__ act,
                                   __nv_bfloat16* __restrict__ dx, int B, int H, int W, int C) {
  const int Ho = H / 2, Wo = W / 2, C8 = C / 8;
  const long n = static_cast<long>(B) * Ho * Wo * C8;
  for (long i = blockIdx.x * static_cast<long>(blockDim.x) + threadIdx.x; i < n;
       i += static_cast<long>(gridDim.x) * blockDim.x) {
    const int c8 = i % C8;
    const int xo = (i / C8) % Wo;
    const int yo = (i / (static_cast<long>(C8) * Wo)) % Ho;
    const int b = i / (static_cast<long>(C8) * Wo * Ho);
    const long base = ((static_cast<long>(b) * H + 2 * yo) * W + 2 * xo) * C + c8 * 8;
    const long offs[4] = {0, C, static_cast<long>(W) * C, static_cast<long>(W) * C + C};
    float a[4][8], g[8];
#pragma unroll
    for (int k = 0; k < 4; ++k) unpack8(__ldg(reinterpret_cast<const uint4*>(act + base + offs[k])), a[k]);
    unpack8(__ldg(reinterpret_cast<const uint4*>(dy + ((static_cast<long>(b) * Ho + yo) * Wo + xo) * C + c8 * 8)), g);
    float o[4][8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      int arg = 0;
      float m = a[0][j];
#pragma unroll
      for (int k = 1; k < 4; ++k)
        if (a[k][j] > m) { m = a[k][j]; arg = k; }
#pragma unroll
      for (int k = 0; k < 4; ++k) o[k][j] = (k == arg && m > 0.f) ? g[j] : 0.f;
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) *reinterpret_cast<uint4*>(dx + base + offs[k]) = pack8(o[k]);
  }
}

int maxpool_bwd(const __nv_bfloat16* dy, const __nv_bfloat16* act, __nv_bfloat16* dx, int B, int H, int W, int C,
                cudaStream_t s) {
  ISX_REQUIRE(C % 8 == 0 && H >= 2 && W >= 2, "maxpool_bwd: bad shape H=%d W=%d C=%d", H, W, C);
  if ((H & 1) || (W & 1))  // the last row / column belongs to no window: gradient 0
    ISX_CHECK_CUDA(cudaMemsetAsync(dx, 0, static_cast<size_t>(B) * H * W * C * 2, s));
  const long n = static_cast<long>(B) * (H / 2) * (W / 2) * (C / 8);
  const int blocks = static_cast<int>(std::min<long>((n + 255) / 256, static_cast<long>(isx_num_sms()) * 16));
  maxpool_bwd_kernel<<<blocks, 256, 0, s>>>(dy, act, dx, B, H, W, C);
  ISX_LAUNCH_CHECK();
  return 0;
}

// The same pool with the routing codes of its backward (pool4_codes: first-maximum position 0..3, 4 = blocked by the ReLU)
// stored as one byte per pooled element -- what the conv epilogues emit when they fuse the pool.  The backward then reads
// the pooled gradient and the codes (3 B per pooled element) instead of the four pre-pool activations (8 B).
__global__ void maxpool_fwd_idx_kernel(const __nv_bfloat16* __restrict__ in, __nv_bfloat16* __restrict__ out,
                                       uint8_t* __restrict__ idx, int B, int H, int W, int C) {
  const int Ho = H / 2, Wo = W / 2, C8 = C / 8;
  const long n = static_cast<long>(B) * Ho * Wo * C8;
  for (long i = blockIdx.x * static_cast<long>(blockDim.x) + threadIdx.x; i < n;
       i += static_cast<long>(gridDim.x) * blockDim.x) {
    const int c8 = i % C8;
    const int xo = (i / C8) % Wo;
    const int yo = (i / (static_cast<long>(C8) * Wo)) % Ho;
    const int b = i / (static_cast<long>(C8) * Wo * Ho);
    const __nv_bfloat16* p = in + ((static_cast<long>(b) * H + 2 * yo) * W + 2 * xo) * C + c8 * 8;
    uint4 u[4];
    u[0] = __ldg(reinterpret_cast<const uint4*>(p));
    u[1] = __ldg(reinterpret_cast<const uint4*>(p + C));
    u[2] = __ldg(reinterpret_cast<const uint4*>(p + static_cast<long>(W) * C));
    u[3] = __ldg(reinterpret_cast<const uint4*>(p + static_cast<long>(W) * C + C));
    uint4 m4;
    uint2 codes;
    pool4_codes(u, m4, codes);
    const long o = ((static_cast<long>(b) * Ho + yo) * Wo + xo) * C + c8 * 8;
    if (out != nullptr) *reinterpret_cast<uint4*>(out + o) = m4;
    *reinterpret_cast<uint2*>(idx + o) = codes;
  }
}

int maxpool_fwd_idx(const __nv_bfloat16* in, __nv_bfloat16* out, uint8_t* idx, int B, int H, int W, int C, cudaStream_t s) {
  ISX_REQUIRE(C % 8 == 0 && H >= 2 && W >= 2, "maxpool: bad shape H=%d W=%d C=%d", H, W, C);
  const long n = static_cast<long>(B) * (H / 2) * (W / 2) * (C / 8);
  const int blocks = static_cast<int>(std::min<long>((n + 255) / 256, static_cast<long>(isx_num_sms()) * 16));
  maxpool_fwd_idx_kernel<<<blocks, 256, 0, s>>>(in, out, idx, B, H, W, C);
  ISX_LAUNCH_CHECK();
  return 0;
}

// dx[pre-pool position k] = (code == k) ? dy[pooled] : 0
__global__ void maxpool_bwd_idx_kernel(const __nv_bfloat16* __restrict__ dy, const uint8_t* __restrict__ idx,
                                       __nv_bfloat16* __restrict__ dx, int B, int H, int W, int C) {
  const int Ho = H / 2, Wo = W / 2, C8 = C / 8;
  const long n = static_cast<long>(B) * Ho * Wo * C8;
  for (long i = blockIdx.x * static_cast<long>(blockDim.x) + threadIdx.x; i < n;
       i += static_cast<long>(gridDim.x) * blockDim.x) {
    const int c8 = i % C8;
    const int xo = (i / C8) % Wo;
    const int yo = (i / (static_cast<long>(C8) * Wo)) % Ho;
    const int b = i / (static_cast<long>(C8) * Wo * Ho);
    const long po = ((static_cast<long>(b) * Ho + yo) * Wo + xo) * C + c8 * 8;
    const uint4 g = __ldg(reinterpret_cast<const uint4*>(dy + po));
    const uint2 cd = __ldg(reinterpret_cast<const uint2*>(idx + po));
    const uint32_t gw[4] = {g.x, g.y, g.z, g.w};
    // codes of elements (2e, 2e+1) as 16-bit lanes: byte 2e of the code word pair -> low half, byte 2e+1 -> high half
    const uint32_t c16[4] = {__byte_perm(cd.x, 0u, 0x4140), __byte_perm(cd.x, 0u, 0x4342), __byte_perm(cd.y, 0u, 0x4140),
                             __byte_perm(cd.y, 0u, 0x4342)};
    const long base = ((static_cast<long>(b) * H + 2 * yo) * W + 2 * xo) * C + c8 * 8;
    const long offs[4] = {0, C, static_cast<long>(W) * C, static_cast<long>(W) * C + C};
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      uint32_t o[4];
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const uint32_t d = c16[e] ^ (static_cast<uint32_t>(k) * 0x00010001u);  // a 16-bit lane is zero where code == k
        const uint32_t keep = ((d & 0x0000FFFFu) ? 0u : 0x0000FFFFu) | ((d & 0xFFFF0000u) ? 0u : 0xFFFF0000u);
        o[e] = gw[e] & keep;
      }
      *reinterpret_cast<uint4*>(dx + base + offs[k]) = make_uint4(o[0], o[1], o[2], o[3]);
    }
  }
}

int maxpool_bwd_idx(const __nv_bfloat16* dy, const uint8_t* idx, __nv_bfloat16* dx, int B, int H, int W, int C,
                    cudaStream_t s) {
  ISX_REQUIRE(C % 8 == 0 && H >= 2 && W >= 2, "maxpool_bwd: bad shape H=%d W=%d C=%d", H, W, C);
  if ((H & 1) || (W & 1))  // the last row / column belongs to no window: gradient 0
    ISX_CHECK_CUDA(cudaMemsetAsync(dx, 0, static_cast<size_t>(B) * H * W * C * 2, s));
  const long n = static_cast<long>(B) * (H / 2) * (W / 2) * (C / 8);
  const int blocks = static_cast<int>(std::min<long>((n + 255) / 256, static_cast<long>(isx_num_sms()) * 16));
  maxpool_bwd_idx_kernel<<<blocks, 256, 0, s>>>(dy, idx, dx, B, H, W, C);
  ISX_LAUNCH_CHECK();
  return 0;
}

// Row G' (mask-weighted Gram, SURVEY.md note N5): Fm = F * m_l (Gram input), Fm2 = F * m_l^2 (its backward operand:
// m * ((F*m) . D) == (F*m^2) . D because m is a per-pixel scalar).  F bf16 [B,HW,C], m fp32 [mask_b,HW].
__global__ void mask_features_kernel(const __nv_bfloat16* __restrict__ f, const float* __restrict__ m, int mask_b,
                                     __nv_bfloat16* __restrict__ fm, __nv_bfloat16* __restrict__ fm2, long HW, int C8,
                                     long n8) {
  for (long i = blockIdx.x * static_cast<long>(blockDim.x) + threadIdx.x; i < n8;
       i += static_cast<long>(gridDim.x) * blockDim.x) {
    const long pix = i / C8;            // b * HW + p
    const long b = pix / HW, pp = pix - b * HW;
    const float mv = __ldg(m + (mask_b > 1 ? b : 0) * HW + pp);
    float a[8], o1[8], o2[8];
    unpack8(__ldg(reinterpret_cast<const uint4*>(f) + i), a);
#pragma unroll
    for (int j = 0; j < 8; ++j) { o1[j] = a[j] * mv; o2[j] = o1[j] * mv; }
    reinterpret_cast<uint4*>(fm)[i] = pack8(o1);
    if (fm2) reinterpret_cast<uint4*>(fm2)[i] = pack8(o2);
  }
}

int mask_features(const __nv_bfloat16* f, const float* m, int mask_b, __nv_bfloat16* fm, __nv_bfloat16* fm2, int B,
                  long HW, int C, cudaStream_t s) {
  const long n8 = static_cast<long>(B) * HW * C / 8;
  const int blocks = static_cast<int>(std::min<long>((n8 + 255) / 256, static_cast<long>(isx_num_sms()) * 16));
  mask_features_kernel<<<blocks, 256, 0, s>>>(f, m, mask_b, fm, fm2, HW, C / 8, n8);
  ISX_LAUNCH_CHECK();
  return 0;
}

// 2x2 stride-2 average pool of an fp32 mask pyramid level: in [B,H,W] -> out [B,H/2,W/2]
__global__ void avgpool2x2_f32_kernel(const float* __restrict__ in, float* __restrict__ out, int B, int H, int W) {
  const int Ho = H / 2, Wo = W / 2;
  const long n = static_cast<long>(B) * Ho * Wo;
  for (long i = blockIdx.x * static_cast<long>(blockDim.x) + threadIdx.x; i < n;
       i += static_cast<long>(gridDim.x) * blockDim.x) {
    const int xo = i % Wo;
    const int yo = (i / Wo) % Ho;
    const long b = i / (static_cast<long>(Wo) * Ho);
    const float* p = in + (b * H + 2 * yo) * W + 2 * xo;
    out[i] = (p[0] + p[1] + p[W] + p[W + 1]) * 0.25f;
  }
}

int avgpool2x2_f32(const float* in, float* out, int B, int H, int W, cudaStream_t s) {
  const long n = static_cast<long>(B) * (H / 2) * (W / 2);
  const int blocks = static_cast<int>(std::min<long>((n + 255) / 256, static_cast<long>(isx_num_sms()) * 8));
  avgpool2x2_f32_kernel<<<blocks, 256, 0, s>>>(in, out, B, H, W);
  ISX_LAUNCH_CHECK();
  return 0;
}

// dx = (g + add) * (act > 0): tap gradient at a layer whose consumer is not a dgrad epilogue
__global__ void tap_add_mask_kernel(const __nv_bfloat16* __restrict__ g, const __nv_bfloat16* __restrict__ add,
                                    const float* __restrict__ aff_a, const float* __restrict__ aff_b,
                                    const __nv_bfloat16* __restrict__ act, __nv_bfloat16* __restrict__ out, long n8,
                                    int C, long per_image8, int relu_mask) {
  for (long i = blockIdx.x * static_cast<long>(blockDim.x) + threadIdx.x; i < n8;
       i += static_cast<long>(gridDim.x) * blockDim.x) {
    float a[8], v[8], t[8];
    unpack8(__ldg(reinterpret_cast<const uint4*>(act) + i), a);
    if (g) unpack8(__ldg(reinterpret_cast<const uint4*>(g) + i), v);
    else {
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] = 0.f;
    }
    if (add) {
      unpack8(__ldg(reinterpret_cast<const uint4*>(add) + i), t);
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] += t[j];
    }
    if (aff_a) {
      const int c = (i * 8) % C;
      const long b = i / per_image8;
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] += aff_a[b * C + c + j] + aff_b[b * C + c + j] * a[j];
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] = (!relu_mask || a[j] > 0.f) ? v[j] : 0.f;
    reinterpret_cast<uint4*>(out)[i] = pack8(v);
  }
}

// Tap gradient of the mask-weighted BN-statistics loss: statistics of Fm = F * m have the affine gradient a + b * Fm w.r.t.
// Fm, hence m * a + m^2 * b * F w.r.t. F (per-pixel weight m, per-(image, channel) a, b)
__global__ void masked_affine_grad_kernel(const __nv_bfloat16* __restrict__ f, const float* __restrict__ m, int mask_b,
                                          const float* __restrict__ aff_a, const float* __restrict__ aff_b,
                                          __nv_bfloat16* __restrict__ out, long HW, int C, long n8) {
  const int C8 = C / 8;
  for (long i = blockIdx.x * static_cast<long>(blockDim.x) + threadIdx.x; i < n8; i += static_cast<long>(gridDim.x) * blockDim.x) {
    const long pix = i / C8;
    const long b = pix / HW, pp = pix - b * HW;
    const int c = static_cast<int>(i % C8) * 8;
    const float mv = __ldg(m + (mask_b > 1 ? b : 0) * HW + pp);
    float a[8], o[8];
    unpack8(__ldg(reinterpret_cast<const uint4*>(f) + i), a);
#pragma unroll
    for (int j = 0; j < 8; ++j) o[j] = mv * (aff_a[b * C + c + j] + aff_b[b * C + c + j] * (mv * a[j]));
    reinterpret_cast<uint4*>(out)[i] = pack8(o);
  }
}

int masked_affine_grad(const __nv_bfloat16* f, const float* m, int mask_b, const float* aff_a, const float* aff_b,
                       __nv_bfloat16* out, int B, long HW, int C, cudaStream_t s) {
  const long n8 = static_cast<long>(B) * HW * C / 8;
  const int blocks = static_cast<int>(std::min<long>((n8 + 255) / 256, static_cast<long>(isx_num_sms()) * 16));
  masked_affine_grad_kernel<<<blocks, 256, 0, s>>>(f, m, mask_b, aff_a, aff_b, out, HW, C, n8);
  ISX_LAUNCH_CHECK();
  return 0;
}

int tap_add_mask(const __nv_bfloat16* g, const __nv_bfloat16* add, const float* aff_a, const float* aff_b,
                 const __nv_bfloat16* act, __nv_bfloat16* out, int B, long HW, int C, cudaStream_t s, int relu_mask) {
  const long n8 = static_cast<long>(B) * HW * C / 8;
  const int blocks = static_cast<int>(std::min<long>((n8 + 255) / 256, static_cast<long>(isx_num_sms()) * 16));
  tap_add_mask_kernel<<<blocks, 256, 0, s>>>(g, add, aff_a, aff_b, act, out, n8, C, HW * C / 8, relu_mask);
  ISX_LAUNCH_CHECK();
  return 0;
}

// ------------------------------------------------------------------------------------------
// Gram finalize: G = sum_splits(partial) * inv_n over the block-upper triangle the symmetric Gram kernel computed
// (128-channel granularity), mirrored into the lower triangle.  One block per 32x32 tile (tr <= tc) of one image.
//   G_out  (optional) full fp32 [B,C,C]
//   loss[b] += loss_scale * sum((G - T)^2)          (StyleLoss_Gram, utils.py:319-321: 0.25 * w_l * sum)
//   D[b]    = grad_scale * (G - T)  in bf16, full     (dF = D . F, see conv_tc 1x1 mode)
//   triu    (optional) upper triangle incl. diagonal in torch.triu_indices order, row b at triu + b * triu_ld
// ------------------------------------------------------------------------------------------
//   kPerProblem: image b belongs to problem p = pw.r.problem_of(b), its gradient scale is (float)(pw.weight[p] * pw.k1 * pw.k2)
//                (beta_p * w_l * inv_n, the same double products the host forms for the scalar grad_scale) and its target
//                is target[pw.target_of(b, p)]
template <bool kPerProblem>
__global__ void __launch_bounds__(256)
gram_finalize_kernel(const float* __restrict__ partial, int splits, int C, float inv_n, float* __restrict__ G_out,
                     const float* __restrict__ target, int target_b, double loss_scale, double* __restrict__ loss,
                     float grad_scale, __nv_bfloat16* __restrict__ D_out, float* __restrict__ triu, long triu_ld,
                     const __grid_constant__ ProblemArg<kPerProblem, ProblemWeights> pw) {
  __shared__ float sg[32][33];
  __shared__ double red[8];
  const int b = blockIdx.y;
  // tile index -> (tr, tc), tr <= tc, row-major over the upper triangle of the nt x nt tile grid
  const int nt = C >> 5;
  int tr = 0, rem = blockIdx.x;
  while (rem >= nt - tr) { rem -= nt - tr; ++tr; }
  const int tc = tr + rem;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const long cc = static_cast<long>(C) * C;
  const float* pb = partial + static_cast<long>(b) * splits * cc;
  const float* tb;
  if constexpr (kPerProblem) {
    const int p = pw.r.problem_of(b);
    tb = target ? target + pw.target_of(b, p) * cc : nullptr;
    grad_scale = static_cast<float>(pw.weight[p] * pw.k1 * pw.k2);
  } else {
    tb = target ? target + (target_b > 1 ? b : 0) * cc : nullptr;
  }
  float d2 = 0.f;
  float g[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const int r = tr * 32 + ty + 8 * k, c = tc * 32 + tx;
    const long o = static_cast<long>(r) * C + c;
    float acc = __ldg(pb + o);
    for (int s = 1; s < splits; ++s) acc += __ldg(pb + s * cc + o);
    g[k] = acc * inv_n;
    sg[ty + 8 * k][tx] = g[k];
    if (G_out) G_out[b * cc + o] = g[k];
    if (triu && c >= r) triu[b * triu_ld + static_cast<long>(r) * C - (static_cast<long>(r) * (r - 1)) / 2 + (c - r)] = g[k];
    if (tb) {
      const float d = g[k] - __ldg(tb + o);
      d2 = fmaf(d, d, d2);
      if (D_out) D_out[b * cc + o] = __float2bfloat16_rn(d * grad_scale);
    }
  }
  if (tr != tc) {  // mirror tile: entry (row, col) = (tc*32 + ty + 8k, tr*32 + tx) = G(tr*32 + tx, tc*32 + ty + 8k)
    __syncthreads();
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const int r = tc * 32 + ty + 8 * k, c = tr * 32 + tx;
      const long o = static_cast<long>(r) * C + c;
      const float v = sg[tx][ty + 8 * k];
      if (G_out) G_out[b * cc + o] = v;
      if (tb) {
        const float d = v - __ldg(tb + o);
        d2 = fmaf(d, d, d2);
        if (D_out) D_out[b * cc + o] = __float2bfloat16_rn(d * grad_scale);
      }
    }
  }
  if (loss) {
    double v = warp_sum(static_cast<double>(d2));
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
    __syncthreads();
    if (threadIdx.x < 32) {
      v = threadIdx.x < 8 ? red[threadIdx.x] : 0.0;
      v = warp_sum(v);
      if (threadIdx.x == 0 && v != 0.0) atomicAdd(loss + b, v * loss_scale);
    }
  }
}

int gram_finalize(const float* partial, int B, int splits, int C, float inv_n, float* G_out, const float* target,
                  int target_b, double loss_scale, double* loss, float grad_scale, __nv_bfloat16* D_out,
                  cudaStream_t s, float* triu, long triu_ld, const ProblemWeights* pw) {
  ISX_REQUIRE(C % 32 == 0, "gram_finalize: C = %d must be a multiple of 32", C);
  const int nt = C / 32;
  dim3 grid(static_cast<unsigned>(nt * (nt + 1) / 2), B);
  if (pw)
    gram_finalize_kernel<true><<<grid, 256, 0, s>>>(partial, splits, C, inv_n, G_out, target, target_b, loss_scale,
                                                    target ? loss : nullptr, grad_scale, D_out, triu, triu_ld, *pw);
  else
    gram_finalize_kernel<false><<<grid, 256, 0, s>>>(partial, splits, C, inv_n, G_out, target, target_b, loss_scale,
                                                     target ? loss : nullptr, grad_scale, D_out, triu, triu_ld, NoProblems());
  ISX_LAUNCH_CHECK();
  return 0;
}

// ------------------------------------------------------------------------------------------
// Content loss (ContentLoss_L2, utils.py:285-290): loss[b] += loss_scale * sum((p-t)^2);
// grad = grad_scale * (p - t) * (p > 0)  (dL/d relu-output, already pushed through the ReLU)
// ------------------------------------------------------------------------------------------
// kPerProblem: image b of problem p = pw.r.problem_of(b) with g_p images has denom = pw.k2 * g_p (per_image * g_p, the
// host's double product for equal problems), loss_scale = 0.5 * pw.k1 / denom and grad_scale = (float)(pw.weight[p] *
// pw.k1 / denom)  (alpha_p * content_w / denom)
template <bool kPerProblem>
__global__ void __launch_bounds__(256)
content_mse_kernel(const __nv_bfloat16* __restrict__ pred, const __nv_bfloat16* __restrict__ target, int target_b,
                   __nv_bfloat16* __restrict__ grad, long per_image8, double loss_scale, float grad_scale,
                   double* __restrict__ loss, int relu_mask, const __grid_constant__ ProblemArg<kPerProblem, ProblemWeights> pw) {
  const int b = blockIdx.y;
  if constexpr (kPerProblem) {
    const int p = pw.r.problem_of(b);
    const double denom = pw.k2 * static_cast<double>(pw.r.size(p));
    loss_scale = 0.5 * pw.k1 / denom;
    grad_scale = static_cast<float>(pw.weight[p] * pw.k1 / denom);
  }
  const uint4* p = reinterpret_cast<const uint4*>(pred) + b * per_image8;
  const uint4* t = reinterpret_cast<const uint4*>(target) + (target_b > 1 ? b : 0) * per_image8;
  uint4* g = grad ? reinterpret_cast<uint4*>(grad) + b * per_image8 : nullptr;
  float acc = 0.f;
  for (long i = blockIdx.x * static_cast<long>(blockDim.x) + threadIdx.x; i < per_image8;
       i += static_cast<long>(gridDim.x) * blockDim.x) {
    float a[8], c[8], o[8];
    unpack8(__ldg(p + i), a);
    unpack8(__ldg(t + i), c);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float d = a[j] - c[j];
      acc = fmaf(d, d, acc);
      o[j] = (!relu_mask || a[j] > 0.f) ? d * grad_scale : 0.f;
    }
    if (g) g[i] = pack8(o);
  }
  __shared__ double red[8];
  double v = warp_sum(static_cast<double>(acc));
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  if (threadIdx.x < 32) {
    v = threadIdx.x < 8 ? red[threadIdx.x] : 0.0;
    v = warp_sum(v);
    if (threadIdx.x == 0) atomicAdd(loss + b, v * loss_scale);
  }
}

int content_mse(const __nv_bfloat16* pred, const __nv_bfloat16* target, int target_b, __nv_bfloat16* grad, int B,
                long per_image, double loss_scale, float grad_scale, double* loss, cudaStream_t s, int relu_mask,
                const ProblemWeights* pw) {
  ISX_REQUIRE(per_image % 8 == 0, "content_mse: per-image size %ld not a multiple of 8", per_image);
  const long n8 = per_image / 8;
  int bx = static_cast<int>(std::min<long>((n8 + 255) / 256, static_cast<long>(isx_num_sms()) * 8 / std::max(1, std::min(B, 8)) + 1));
  dim3 grid(bx, B);
  if (pw)
    content_mse_kernel<true><<<grid, 256, 0, s>>>(pred, target, target_b, grad, n8, loss_scale, grad_scale, loss, relu_mask, *pw);
  else
    content_mse_kernel<false><<<grid, 256, 0, s>>>(pred, target, target_b, grad, n8, loss_scale, grad_scale, loss, relu_mask,
                                                   NoProblems());
  ISX_LAUNCH_CHECK();
  return 0;
}

// ------------------------------------------------------------------------------------------
// Per-(image, channel) sum and sum of squares over H*W  (StyleLoss_BN utils.py:337-338, 350-352;
// Classifier2 features classifiers.py:71).  sums[b][c][2] (double) must be zeroed by the caller.
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
chan_sums_kernel(const __nv_bfloat16* __restrict__ f, long HW, int C, double* __restrict__ sums,
                 const float* __restrict__ mask, int mask_b) {
  extern __shared__ float sred[];  // [256][16]
  const int b = blockIdx.y;
  const int C8 = C / 8;
  const int lanes = 256 / C8;          // pixel lanes per block (C8 <= 64)
  const int c8 = threadIdx.x % C8;
  const int pl = threadIdx.x / C8;
  float s1[8], s2[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) s1[j] = s2[j] = 0.f;
  if (pl < lanes) {
    const uint4* base = reinterpret_cast<const uint4*>(f + static_cast<long>(b) * HW * C) + c8;
    for (long p = blockIdx.x * static_cast<long>(lanes) + pl; p < HW; p += static_cast<long>(gridDim.x) * lanes) {
      float a[8];
      unpack8(__ldg(base + p * C8), a);
      if (mask) {   // statistics of F * m (mask-weighted BN loss): per-pixel weight
        const float mv = __ldg(mask + (mask_b > 1 ? b : 0) * HW + p);
#pragma unroll
        for (int j = 0; j < 8; ++j) a[j] *= mv;
      }
#pragma unroll
      for (int j = 0; j < 8; ++j) { s1[j] += a[j]; s2[j] = fmaf(a[j], a[j], s2[j]); }
    }
  }
#pragma unroll
  for (int j = 0; j < 8; ++j) { sred[threadIdx.x * 16 + j] = s1[j]; sred[threadIdx.x * 16 + 8 + j] = s2[j]; }
  __syncthreads();
  // thread t < C8*16 reduces one (c8, slot) over pixel lanes
  for (int t = threadIdx.x; t < C8 * 16; t += blockDim.x) {
    const int cc8 = t / 16, slot = t % 16;
    double acc = 0.0;
    for (int l = 0; l < lanes; ++l) acc += static_cast<double>(sred[(l * C8 + cc8) * 16 + slot]);
    const int c = cc8 * 8 + (slot & 7);
    atomicAdd(sums + (static_cast<long>(b) * C + c) * 2 + (slot >> 3), acc);
  }
}

int chan_sums(const __nv_bfloat16* f, int B, long HW, int C, double* sums, cudaStream_t s, const float* mask, int mask_b) {
  ISX_REQUIRE(C % 8 == 0 && C / 8 <= 64 && 256 % (C / 8) == 0, "chan_sums: C=%d unsupported", C);
  const int lanes = 256 / (C / 8);
  long bx = (HW + lanes * 8 - 1) / (lanes * 8);  // >= 8 pixels per lane
  const long cap = std::max<long>(1, static_cast<long>(isx_num_sms()) * 4 / B);
  if (bx > cap) bx = cap;
  if (bx < 1) bx = 1;
  dim3 grid(static_cast<unsigned>(bx), B);
  chan_sums_kernel<<<grid, 256, 256 * 16 * sizeof(float), s>>>(f, HW, C, sums, mask, mask_b);
  ISX_LAUNCH_CHECK();
  return 0;
}

// mean / unbiased std from the sums; optional StyleLoss_BN loss + affine tap-gradient coefficients:
//   loss[b] += loss_scale * sum_c[(mu-mu_t)^2 + (sd-sd_t)^2]            (loss_scale = w_l / C)
//   dL/dF[p,c] = aff_a[b,c] + aff_b[b,c] * F[p,c]   with (grad_scale = beta * w_l / C)
//     aff_b = grad_scale * 2 (sd - sd_t) / ((n-1) sd),  aff_a = grad_scale * 2 (mu - mu_t) / n - aff_b * mu
// kPerProblem: image b of problem p = pw.r.problem_of(b): grad_scale = pw.weight[p] * pw.k1 / pw.k2  (beta_p * w_l / C),
// target pw.target_of(b, p)
template <bool kPerProblem>
__global__ void bn_finalize_kernel(const double* __restrict__ sums, int B, int C, double n, float* __restrict__ mean,
                                   float* __restrict__ stdv, const float* __restrict__ t_mean,
                                   const float* __restrict__ t_std, int target_b, double loss_scale, double grad_scale,
                                   double* __restrict__ loss, float* __restrict__ aff_a, float* __restrict__ aff_b,
                                   long out_ld, const __grid_constant__ ProblemArg<kPerProblem, ProblemWeights> pw) {
  const int b = blockIdx.x;
  int tp = 0;   // the image's style target row
  if constexpr (kPerProblem) {
    const int p = pw.r.problem_of(b);
    grad_scale = pw.weight[p] * pw.k1 / pw.k2;
    tp = pw.target_of(b, p);
  }
  double lacc = 0.0;
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    const double s1 = sums[(static_cast<long>(b) * C + c) * 2], s2 = sums[(static_cast<long>(b) * C + c) * 2 + 1];
    const double mu = s1 / n;
    double var = (s2 - s1 * mu) / (n - 1.0);
    if (var < 0.0) var = 0.0;
    const double sd = sqrt(var);
    if (mean) mean[b * out_ld + c] = static_cast<float>(mu);
    if (stdv) stdv[b * out_ld + c] = static_cast<float>(sd);
    if (t_mean) {
      const int tb = kPerProblem ? tp : (target_b > 1 ? b : 0);
      const double dm = static_cast<double>(static_cast<float>(mu)) - t_mean[tb * C + c];
      const double ds = static_cast<double>(static_cast<float>(sd)) - t_std[tb * C + c];
      lacc += dm * dm + ds * ds;
      if (aff_a) {
        const double bb = sd > 0.0 ? grad_scale * 2.0 * ds / ((n - 1.0) * sd) : 0.0;
        aff_b[b * C + c] = static_cast<float>(bb);
        aff_a[b * C + c] = static_cast<float>(grad_scale * 2.0 * dm / n - bb * mu);
      }
    }
  }
  if (loss && t_mean) {
    __shared__ double red[8];
    double v = warp_sum(lacc);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
    __syncthreads();
    if (threadIdx.x < 32) {
      v = threadIdx.x < (blockDim.x >> 5) ? red[threadIdx.x] : 0.0;
      v = warp_sum(v);
      if (threadIdx.x == 0) atomicAdd(loss + b, v * loss_scale);
    }
  }
}

// mean / unbiased std from what the Gram kernel left behind: S1 = sum over splits of its fused channel sums, S2 = sum over
// splits of the diagonal of the raw Gram partials (sum of squares); double arithmetic from here on
__global__ void stats_from_gram_kernel(const float* __restrict__ partial, const float* __restrict__ csum, int splits, int C,
                                       double n, float* __restrict__ mean, float* __restrict__ stdv, long out_ld) {
  const int b = blockIdx.x;
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    double s1 = 0.0, s2 = 0.0;
    for (int s = 0; s < splits; ++s) {
      s1 += static_cast<double>(csum[(static_cast<long>(b) * splits + s) * C + c]);
      s2 += static_cast<double>(partial[((static_cast<long>(b) * splits + s) * C + c) * C + c]);
    }
    const double mu = s1 / n;
    double var = (s2 - s1 * mu) / (n - 1.0);
    if (var < 0.0) var = 0.0;
    mean[b * out_ld + c] = static_cast<float>(mu);
    stdv[b * out_ld + c] = static_cast<float>(sqrt(var));
  }
}

int stats_from_gram(const float* partial, const float* csum, int B, int splits, int C, long HW, float* mean, float* stdv,
                    long out_ld, cudaStream_t s) {
  stats_from_gram_kernel<<<B, 128, 0, s>>>(partial, csum, splits, C, static_cast<double>(HW), mean, stdv, out_ld);
  ISX_LAUNCH_CHECK();
  return 0;
}

int bn_finalize(const double* sums, int B, int C, long HW, float* mean, float* stdv, const float* t_mean,
                const float* t_std, int target_b, double loss_scale, double grad_scale, double* loss, float* aff_a,
                float* aff_b, cudaStream_t s, long out_ld, const ProblemWeights* pw) {
  if (pw)
    bn_finalize_kernel<true><<<B, 256, 0, s>>>(sums, B, C, static_cast<double>(HW), mean, stdv, t_mean, t_std, target_b,
                                               loss_scale, grad_scale, loss, aff_a, aff_b, out_ld > 0 ? out_ld : C, *pw);
  else
    bn_finalize_kernel<false><<<B, 256, 0, s>>>(sums, B, C, static_cast<double>(HW), mean, stdv, t_mean, t_std, target_b,
                                                loss_scale, grad_scale, loss, aff_a, aff_b, out_ld > 0 ? out_ld : C,
                                                NoProblems());
  ISX_LAUNCH_CHECK();
  return 0;
}

}  // namespace isx
