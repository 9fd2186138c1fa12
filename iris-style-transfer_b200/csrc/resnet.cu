// ResNet-50 trunk (torchvision resnet50 in eval mode, the feature extractor of GazeEstimator2: reference
// models/gaze_estimators/gaze_estimators.py:180-223 with models/resnet/resnet.py) on the device:
//   * the 7x7 / stride 2 / pad 3 stem (3 -> 64) + bias + ReLU as one tcgen05 MMA chain per 128 output pixels, gathered
//     straight from the fp32 NCHW image (K = 147 taps padded to 192 = three 64-wide K blocks);
//   * MaxPool2d(3, 2, 1) over bf16 NHWC (padding = -inf, torch's first-maximum rule: bit-exact);
//   * the global average pool bf16 NHWC [B,h,w,C] -> fp32 [B,C] (fp64 partial sums, fixed order: deterministic);
//   * the bottlenecks on the generic implicit-GEMM conv (conv_tc.cu: 1x1 and 3x3, stride 1 or 2, bias + residual + ReLU);
//   * isx_resnet50_forward chaining the 53 convolutions through five rotating activation buffers.
// BatchNorm is folded into the convolutions by the caller (eval mode), so every conv is conv + bias.
#include <algorithm>

#include "../../include/isx.h"
#include "isx_common.cuh"
#include "isx_internal.h"
#include "isx_kernels.h"

namespace isx {

typedef __nv_bfloat16 bf16;

// ---------------------------------------------------------------------------------------------
// weight packing
// ---------------------------------------------------------------------------------------------
__global__ void to_bf16_kernel(const float* __restrict__ w, bf16* __restrict__ out, long n) {
  const long i = static_cast<long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i < n) out[i] = __float2bfloat16_rn(w[i]);
}

// fp32 OIHW [64,3,7,7] -> bf16 [64][192]: K index = c*49 + ky*7 + kx (the OIHW order), 147..191 zero
__global__ void pack_stem_kernel(const float* __restrict__ w, bf16* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= 64 * 192) return;
  const int k = i % 192, o = i / 192;
  out[i] = __float2bfloat16_rn(k < 147 ? w[o * 147 + k] : 0.f);
}

// ---------------------------------------------------------------------------------------------
// stem: 7x7 s2 p3 conv (3 -> 64) + bias + ReLU on tcgen05
// ---------------------------------------------------------------------------------------------
static constexpr int kStemK = 192;                       // 147 taps padded to three 64-wide K blocks
static constexpr int kStemA = 3 * 16384;                 // A: 3 K blocks x 128 rows x 128 B (SWIZZLE_128B, K-major)
static constexpr int kStemB = 3 * 8192;                  // B: 3 K blocks x 64 rows x 128 B
static constexpr int kStemBar = kStemA + kStemB;         // barriers + TMEM address
static constexpr int kStemBias = kStemBar + 64;
static constexpr int kStemPatch = kStemBias + 256;       // bf16 [3][2TH+5][2TW+5] input patch of the tile

struct StemParams {
  const float* x;
  const float* bias;
  int xc, B, H, W, Ho, Wo;
  int TW, TH, tiles_x, tiles_y, n_tiles;
};

template <int TW>
__global__ void __launch_bounds__(128, 2)
resnet_stem_kernel(const __grid_constant__ CUtensorMap tmW, const __grid_constant__ CUtensorMap tmO, const StemParams p) {
  constexpr int TH = 128 / TW;
  constexpr int PW = 2 * TW + 5, PH = 2 * TH + 5;
  constexpr int npatch = 3 * PH * PW;
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* sA = smem;
  uint8_t* sB = smem + kStemA;
  uint8_t* sO = sA;  // output staging aliases the first A block (free once the MMAs have completed)
  uint64_t* w_bar = reinterpret_cast<uint64_t*>(smem + kStemBar);
  uint64_t* mma_bar = w_bar + 1;
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(mma_bar + 1);
  float* s_bias = reinterpret_cast<float*>(smem + kStemBias);
  bf16* s_patch = reinterpret_cast<bf16*>(smem + kStemPatch);
  const int tid = threadIdx.x, warp = tid >> 5;

  if (tid == 0) {
    if (smem_u32(smem) & 1023u) {
      printf("isx: resnet stem: dynamic shared memory is not 1024-byte aligned\n");
      __trap();
    }
    tma_prefetch_desc(&tmW);
    tma_prefetch_desc(&tmO);
    mbar_init(w_bar, 1);
    mbar_init(mma_bar, 1);
    fence_barrier_init();
  }
  if (tid < 64) s_bias[tid] = p.bias ? p.bias[tid] : 0.f;
  if (warp == 0) tmem_alloc<64>(tmem_ptr_smem);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;
  if (tid == 0) {
    mbar_arrive_expect_tx(w_bar, kStemB);
#pragma unroll
    for (int kb = 0; kb < 3; ++kb) tma_load_2d(sB + kb * 8192, &tmW, w_bar, kb * 64, 0);
  }
  const long hw = static_cast<long>(p.H) * p.W;
  constexpr uint32_t idesc = umma_idesc_bf16(128, 64, false, false);
  uint32_t phase = 0;
  bool w_ready = false;
  const int tw = tid % TW, th = tid / TW;
  for (int tile = blockIdx.x; tile < p.n_tiles; tile += gridDim.x) {
    const int tx = tile % p.tiles_x;
    const int ty = (tile / p.tiles_x) % p.tiles_y;
    const int b = tile / (p.tiles_x * p.tiles_y);
    const int x0 = tx * TW, y0 = ty * TH;
    // ---- input patch of the tile -> bf16 in shared memory (zero padding) ----
    for (int i = tid; i < npatch; i += 128) {
      const int px = i % PW;
      const int py = (i / PW) % PH;
      const int c = i / (PW * PH);
      const int y = 2 * y0 + py - 3, xq = 2 * x0 + px - 3;
      float v = 0.f;
      if (y >= 0 && y < p.H && xq >= 0 && xq < p.W)
        v = __ldg(p.x + (static_cast<long>(b) * p.xc + (p.xc == 3 ? c : 0)) * hw + static_cast<long>(y) * p.W + xq);
      s_patch[i] = __float2bfloat16_rn(v);
    }
    if (tid == 0) tma_store_wait_read<0>();  // the previous tile's TMA store has finished reading sA (== staging)
    __syncthreads();
    // ---- this thread's output pixel: 147 taps -> one 384-byte K-major row over the three swizzled A blocks ----
    const bf16* pp = s_patch + (2 * th) * PW + 2 * tw;
    uint8_t* rowp = sA + tid * 128;
#pragma unroll
    for (int kb = 0; kb < 3; ++kb) {
#pragma unroll
      for (int ch = 0; ch < 8; ++ch) {
        uint32_t wd[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          uint32_t pair = 0;
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            const int k = kb * 64 + ch * 8 + j * 2 + h;
            if (k < 147) {
              const int c = k / 49, ky = (k % 49) / 7, kx = k % 7;
              pair |= static_cast<uint32_t>(__bfloat16_as_ushort(pp[(c * PH + ky) * PW + kx])) << (16 * h);
            }
          }
          wd[j] = pair;
        }
        *reinterpret_cast<uint4*>(rowp + kb * 16384 + ((ch ^ (tid & 7)) * 16)) = make_uint4(wd[0], wd[1], wd[2], wd[3]);
      }
    }
    fence_proxy_async_smem();  // generic-proxy smem writes -> visible to the tensor core (async proxy)
    __syncthreads();
    if (tid == 0) {
      if (!w_ready) mbar_wait(w_bar, 0);
      tc_fence_after();
      const uint32_t a_addr = smem_u32(sA), b_addr = smem_u32(sB);
#pragma unroll
      for (int kb = 0; kb < 3; ++kb)
#pragma unroll
        for (int k = 0; k < 4; ++k)
          umma_bf16(tmem_base, umma_desc_sw128(a_addr + kb * 16384 + k * 32, 16, 1024),
                    umma_desc_sw128(b_addr + kb * 8192 + k * 32, 16, 1024), idesc, (kb | k) != 0 ? 1u : 0u);
      umma_commit(mma_bar);
    }
    w_ready = true;
    mbar_wait(mma_bar, phase);
    phase ^= 1;
    tc_fence_after();
    // ---- epilogue: bias + ReLU -> bf16 -> swizzled staging -> TMA store ----
#pragma unroll 1
    for (int hlf = 0; hlf < 2; ++hlf) {
      uint32_t v[32];
      tmem_ld_32x32(tmem_base + (static_cast<uint32_t>(warp * 32) << 16) + hlf * 32, v);
      tmem_ld_wait();
      uint8_t* orow = sO + tid * 128;
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        float f[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) f[j] = fmaxf(__uint_as_float(v[c * 8 + j]) + s_bias[hlf * 32 + c * 8 + j], 0.f);
        uint4 o;
        o.x = pack_bf16x2(f[0], f[1]); o.y = pack_bf16x2(f[2], f[3]);
        o.z = pack_bf16x2(f[4], f[5]); o.w = pack_bf16x2(f[6], f[7]);
        *reinterpret_cast<uint4*>(orow + (((hlf * 4 + c) ^ (tid & 7)) * 16)) = o;
      }
    }
    fence_proxy_async_smem();
    tc_fence_before();
    __syncthreads();
    if (tid == 0) {
      tma_store_4d(&tmO, sO, 0, x0, y0, b);
      tma_store_commit();
    }
  }
  if (tid == 0) tma_store_wait_all<0>();
  __syncthreads();
  if (warp == 0) {
    tc_fence_after();
    tmem_dealloc<64>(tmem_base);
  }
}

static int resnet_stem(const float* x, int xc, const bf16* w_packed, const float* bias, bf16* out, int B, int H, int W,
                       cudaStream_t s) {
  ISX_REQUIRE(xc == 1 || xc == 3, "resnet stem: image must have 1 or 3 channels, got %d", xc);
  StemParams p;
  p.x = x; p.bias = bias; p.xc = xc; p.B = B; p.H = H; p.W = W;
  p.Ho = (H + 1) / 2; p.Wo = (W + 1) / 2;
  // 128-pixel tile with the least work: padded output pixels x the size of its (2TW+5) x (2TH+5) input patch
  double best = -1.0;
  for (int twc = 128; twc >= 1; twc >>= 1) {
    const int thc = 128 / twc;
    const double padded = static_cast<double>((p.Wo + twc - 1) / twc * twc) * ((p.Ho + thc - 1) / thc * thc);
    const double cost = padded * ((2 * twc + 5) * (2 * thc + 5));
    if (best < 0 || cost < best) { best = cost; p.TW = twc; p.TH = thc; }
  }
  p.tiles_x = (p.Wo + p.TW - 1) / p.TW;
  p.tiles_y = (p.Ho + p.TH - 1) / p.TH;
  const long nt = static_cast<long>(p.tiles_x) * p.tiles_y * B;
  ISX_REQUIRE(nt < (1L << 31), "resnet stem: too many tiles");
  p.n_tiles = static_cast<int>(nt);
  CUtensorMap tmW, tmO;
  {
    uint64_t dims[2] = {kStemK, 64};
    uint64_t str[1] = {kStemK * 2};
    uint32_t box[2] = {64, 64};
    if (isx_make_tmap_bf16(&tmW, w_packed, 2, dims, str, box, true)) return 3;
  }
  {
    uint64_t dims[4] = {64, (uint64_t)p.Wo, (uint64_t)p.Ho, (uint64_t)B};
    uint64_t str[3] = {128, (uint64_t)p.Wo * 128, (uint64_t)p.Ho * p.Wo * 128};
    uint32_t box[4] = {64, (uint32_t)p.TW, (uint32_t)p.TH, 1};
    if (isx_make_tmap_bf16(&tmO, out, 4, dims, str, box, true)) return 3;
  }
  const size_t smem_bytes = kStemPatch + 2 * 3 * (2 * p.TW + 5) * (2 * p.TH + 5);
  const int grid = std::min(p.n_tiles, kNumSMs * 16);
  isx_prof_begin(ISX_PROF_CONV, 2.0 * 147 * 64 * static_cast<double>(B) * p.Ho * p.Wo, s);
#define ISX_STEM_CASE(TW_)                                                                                                   \
  case TW_:                                                                                                                  \
    ISX_CHECK_CUDA(cudaFuncSetAttribute(resnet_stem_kernel<TW_>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bytes)); \
    resnet_stem_kernel<TW_><<<grid, 128, smem_bytes, s>>>(tmW, tmO, p);                                                      \
    break;
  switch (p.TW) {
    ISX_STEM_CASE(128) ISX_STEM_CASE(64) ISX_STEM_CASE(32) ISX_STEM_CASE(16) ISX_STEM_CASE(8) ISX_STEM_CASE(4)
    ISX_STEM_CASE(2) ISX_STEM_CASE(1)
    default: ISX_REQUIRE(false, "resnet stem: bad tile width %d", p.TW);
  }
#undef ISX_STEM_CASE
  isx_prof_end(ISX_PROF_CONV, s);
  ISX_LAUNCH_CHECK();
  return 0;
}

// ---------------------------------------------------------------------------------------------
// MaxPool2d(kernel 3, stride 2, padding 1) over bf16 NHWC; one thread per output pixel and 8 channels (128-bit accesses)
// ---------------------------------------------------------------------------------------------
__global__ void maxpool3x3s2_kernel(const bf16* __restrict__ in, bf16* __restrict__ out, int H, int W, int C, int Ho, int Wo,
                                    long n) {
  const long i = static_cast<long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int C8 = C >> 3;
  const int c8 = static_cast<int>(i % C8);
  long r = i / C8;
  const int xo = static_cast<int>(r % Wo);
  r /= Wo;
  const int yo = static_cast<int>(r % Ho);
  const long b = r / Ho;
  float m[8];
  unsigned short mb[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) { m[j] = -INFINITY; mb[j] = 0xFF80u; }  // bf16 -inf
  // window scan in torch's order with its rule (val > max || isnan(val)): the first maximum wins, NaN propagates
  for (int dy = -1; dy <= 1; ++dy) {
    const int y = 2 * yo + dy;
    if (y < 0 || y >= H) continue;
    for (int dx = -1; dx <= 1; ++dx) {
      const int x = 2 * xo + dx;
      if (x < 0 || x >= W) continue;
      const uint4 u = __ldg(reinterpret_cast<const uint4*>(in + ((b * H + y) * W + x) * C) + c8);
      const unsigned short* e = reinterpret_cast<const unsigned short*>(&u);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float v = __uint_as_float(static_cast<uint32_t>(e[j]) << 16);
        if (v > m[j] || isnan(v)) { m[j] = v; mb[j] = e[j]; }
      }
    }
  }
  uint4 o;
  o.x = mb[0] | (static_cast<uint32_t>(mb[1]) << 16);
  o.y = mb[2] | (static_cast<uint32_t>(mb[3]) << 16);
  o.z = mb[4] | (static_cast<uint32_t>(mb[5]) << 16);
  o.w = mb[6] | (static_cast<uint32_t>(mb[7]) << 16);
  reinterpret_cast<uint4*>(out + ((b * Ho + yo) * Wo + xo) * C)[c8] = o;
}

static int maxpool3x3s2(const bf16* in, bf16* out, int B, int H, int W, int C, cudaStream_t s) {
  ISX_REQUIRE(B > 0 && H > 0 && W > 0 && C > 0 && C % 8 == 0, "maxpool3x3s2: bad shape B=%d H=%d W=%d C=%d", B, H, W, C);
  const int Ho = (H + 1) / 2, Wo = (W + 1) / 2;
  const long n = static_cast<long>(B) * Ho * Wo * (C / 8);
  maxpool3x3s2_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, s>>>(in, out, H, W, C, Ho, Wo, n);
  ISX_LAUNCH_CHECK();
  return 0;
}

// ---------------------------------------------------------------------------------------------
// global average pool: bf16 [B,HW,C] -> fp32 [B,C].  Block (32 channel groups of 8) x (8 pixel lanes) per image and
// 256 channels; fp64 partial sums reduced in a fixed order (no atomics: every run gives the same bits).
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) global_avgpool_kernel(const bf16* __restrict__ in, float* __restrict__ out, int HW, int C) {
  __shared__ double part[8][32][8];
  const int cg = threadIdx.x & 31, lane_p = threadIdx.x >> 5;
  const int b = blockIdx.y;
  const int c0 = (blockIdx.x * 32 + cg) * 8;
  double acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  if (c0 < C) {
    const bf16* base = in + static_cast<long>(b) * HW * C + c0;
    for (int pix = lane_p; pix < HW; pix += 8) {
      const uint4 u = __ldg(reinterpret_cast<const uint4*>(base + static_cast<long>(pix) * C));
      const uint32_t w4[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float2 f = unpack_bf16x2(w4[j]);
        acc[2 * j] += f.x;
        acc[2 * j + 1] += f.y;
      }
    }
  }
#pragma unroll
  for (int j = 0; j < 8; ++j) part[lane_p][cg][j] = acc[j];
  __syncthreads();
  if (lane_p == 0 && c0 < C) {
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      double sum = 0.0;
#pragma unroll
      for (int l = 0; l < 8; ++l) sum += part[l][cg][j];
      out[static_cast<long>(b) * C + c0 + j] = static_cast<float>(sum / HW);
    }
  }
}

static int global_avgpool(const bf16* in, float* out, int B, int HW, int C, cudaStream_t s) {
  ISX_REQUIRE(B > 0 && HW > 0 && C > 0 && C % 8 == 0, "global_avgpool: bad shape B=%d HW=%d C=%d", B, HW, C);
  global_avgpool_kernel<<<dim3((C / 8 + 31) / 32, B), 256, 0, s>>>(in, out, HW, C);
  ISX_LAUNCH_CHECK();
  return 0;
}

static int conv_fwd(const bf16* in, const bf16* w, const float* bias, const bf16* residual, bf16* out, int B, int H, int W,
                    int Cin, int Cout, int k, int stride, int relu, cudaStream_t s) {
  ISX_REQUIRE(k == 1 || k == 3, "conv: kernel size %d (1 or 3)", k);
  ISX_REQUIRE(stride == 1 || stride == 2, "conv: stride %d (1 or 2)", stride);
  ConvArgs a;
  a.in = in; a.weight = w; a.out = out; a.bias = bias; a.add_buf = residual; a.relu = relu;
  a.B = B; a.H = H; a.W = W; a.Cin = Cin; a.Cout = Cout; a.ntaps = k * k; a.stride = stride;
  a.generic_only = true;
  return conv_tc(a, s);
}

// ---------------------------------------------------------------------------------------------
// the trunk: shapes and buffers
// ---------------------------------------------------------------------------------------------
static const int kStagePlanes[4] = {64, 128, 256, 512};
static const int kStageBlocks[4] = {3, 4, 6, 3};

struct ResnetPlan {
  // element counts PER IMAGE of the five rotating buffers: block input / output (X, Y), conv1 / conv2 outputs (T1, T2),
  // projection shortcut (D)
  long x, y, t1, t2, d;
};

static ResnetPlan resnet_plan(int H, int W) {
  ResnetPlan pl{0, 0, 0, 0, 0};
  int h = (H + 1) / 2, w = (W + 1) / 2;  // stem
  pl.y = static_cast<long>(h) * w * 64;   // the stem writes Y, the max pool reads it into X
  h = (h + 1) / 2; w = (w + 1) / 2;
  pl.x = static_cast<long>(h) * w * 64;
  for (int st = 0; st < 4; ++st) {
    const int planes = kStagePlanes[st];
    for (int blk = 0; blk < kStageBlocks[st]; ++blk) {
      const int stride = (st > 0 && blk == 0) ? 2 : 1;
      pl.t1 = std::max(pl.t1, static_cast<long>(h) * w * planes);
      const int ho = (h + stride - 1) / stride, wo = (w + stride - 1) / stride;
      const long outn = static_cast<long>(ho) * wo * planes * 4;
      pl.t2 = std::max(pl.t2, static_cast<long>(ho) * wo * planes);
      if (blk == 0) pl.d = std::max(pl.d, outn);
      pl.x = std::max(pl.x, outn);
      pl.y = std::max(pl.y, outn);
      h = ho; w = wo;
    }
  }
  return pl;
}

static int64_t align256(int64_t n) { return (n + 255) & ~static_cast<int64_t>(255); }

}  // namespace isx

using namespace isx;

static inline cudaStream_t S(isx_stream s) { return reinterpret_cast<cudaStream_t>(s); }
static inline const bf16* P(const isx_bf16* p) { return reinterpret_cast<const bf16*>(p); }
static inline bf16* P(isx_bf16* p) { return reinterpret_cast<bf16*>(p); }

extern "C" int isx_pack_conv1x1_weights(const float* w, int Cout, int Cin, isx_bf16* w_out, isx_stream stream) {
  ISX_REQUIRE(w && w_out && Cout > 0 && Cin > 0, "isx_pack_conv1x1_weights: bad arguments");
  const long n = static_cast<long>(Cout) * Cin;
  to_bf16_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, S(stream)>>>(w, P(w_out), n);
  ISX_LAUNCH_CHECK();
  return 0;
}

extern "C" int isx_pack_resnet_stem_weights(const float* w, isx_bf16* w_out, isx_stream stream) {
  ISX_REQUIRE(w && w_out, "isx_pack_resnet_stem_weights: null pointer");
  pack_stem_kernel<<<(64 * 192 + 255) / 256, 256, 0, S(stream)>>>(w, P(w_out));
  ISX_LAUNCH_CHECK();
  return 0;
}

extern "C" int isx_conv_bias_act_fwd(const isx_bf16* in, const isx_bf16* w, const float* bias, const isx_bf16* residual,
                                     isx_bf16* out, int B, int H, int W, int Cin, int Cout, int k, int stride, int relu,
                                     isx_stream stream) {
  ISX_REQUIRE(in && w && out && B > 0 && H > 0 && W > 0, "isx_conv_bias_act_fwd: bad arguments");
  return conv_fwd(P(in), P(w), bias, P(residual), P(out), B, H, W, Cin, Cout, k, stride, relu, S(stream));
}

extern "C" int isx_resnet_stem_fwd(const float* x, int xc, const isx_bf16* w, const float* bias, isx_bf16* out, int B, int H,
                                   int W, isx_stream stream) {
  ISX_REQUIRE(x && w && out && B > 0 && H > 0 && W > 0, "isx_resnet_stem_fwd: bad arguments");
  return resnet_stem(x, xc, P(w), bias, P(out), B, H, W, S(stream));
}

extern "C" int isx_maxpool3x3s2_fwd(const isx_bf16* in, isx_bf16* out, int B, int H, int W, int C, isx_stream stream) {
  ISX_REQUIRE(in && out, "isx_maxpool3x3s2_fwd: null pointer");
  return maxpool3x3s2(P(in), P(out), B, H, W, C, S(stream));
}

extern "C" int isx_global_avgpool(const isx_bf16* in, float* out, int B, int HW, int C, isx_stream stream) {
  ISX_REQUIRE(in && out, "isx_global_avgpool: null pointer");
  return global_avgpool(P(in), out, B, HW, C, S(stream));
}

extern "C" int64_t isx_resnet50_workspace_bytes(int B, int H, int W) {
  if (B <= 0 || H < 32 || W < 32) {
    isx_set_error("isx_resnet50_workspace_bytes: bad shape B=%d H=%d W=%d (B >= 1, H and W >= 32)", B, H, W);
    return -1;
  }
  const ResnetPlan pl = resnet_plan(H, W);
  return align256(pl.x * 2 * B) + align256(pl.y * 2 * B) + align256(pl.t1 * 2 * B) + align256(pl.t2 * 2 * B) +
         align256(pl.d * 2 * B);
}

extern "C" int isx_resnet50_forward(const isx_resnet50_weights* wts, const float* x, int xc, int B, int H, int W,
                                    void* workspace, float* feat_out, isx_stream stream) {
  ISX_REQUIRE(wts && x && workspace && feat_out, "isx_resnet50_forward: null pointer");
  ISX_REQUIRE(B > 0 && H >= 32 && W >= 32, "isx_resnet50_forward: bad shape B=%d H=%d W=%d (H and W >= 32)", B, H, W);
  ISX_REQUIRE(xc == 1 || xc == 3, "isx_resnet50_forward: xc must be 1 or 3, got %d", xc);
  for (int i = 0; i < ISX_RESNET50_CONVS; ++i)
    ISX_REQUIRE(wts->w[i] && wts->bias[i], "isx_resnet50_forward: weights of conv %d missing", i);
  const cudaStream_t s = S(stream);
  const ResnetPlan pl = resnet_plan(H, W);
  uint8_t* ws = static_cast<uint8_t*>(workspace);
  bf16* X = reinterpret_cast<bf16*>(ws);
  ws += align256(pl.x * 2 * B);
  bf16* Y = reinterpret_cast<bf16*>(ws);
  ws += align256(pl.y * 2 * B);
  bf16* T1 = reinterpret_cast<bf16*>(ws);
  ws += align256(pl.t1 * 2 * B);
  bf16* T2 = reinterpret_cast<bf16*>(ws);
  ws += align256(pl.t2 * 2 * B);
  bf16* D = reinterpret_cast<bf16*>(ws);

  int rc = resnet_stem(x, xc, P(wts->w[0]), wts->bias[0], Y, B, H, W, s);
  if (rc) return rc;
  int h = (H + 1) / 2, w = (W + 1) / 2;
  if ((rc = maxpool3x3s2(Y, X, B, h, w, 64, s))) return rc;
  h = (h + 1) / 2; w = (w + 1) / 2;
  int cin = 64, li = 1;
  for (int st = 0; st < 4; ++st) {
    const int planes = kStagePlanes[st], cout = planes * 4;
    for (int blk = 0; blk < kStageBlocks[st]; ++blk) {
      const int stride = (st > 0 && blk == 0) ? 2 : 1;
      const int ho = (h + stride - 1) / stride, wo = (w + stride - 1) / stride;
      // Bottleneck (torchvision v1.5): relu(bn3(conv3(relu(bn2(conv2_s(relu(bn1(conv1(x)))))))) + shortcut(x))
      if ((rc = conv_fwd(X, P(wts->w[li]), wts->bias[li], nullptr, T1, B, h, w, cin, planes, 1, 1, 1, s))) return rc;
      if ((rc = conv_fwd(T1, P(wts->w[li + 1]), wts->bias[li + 1], nullptr, T2, B, h, w, planes, planes, 3, stride, 1, s)))
        return rc;
      const bf16* shortcut = X;
      if (blk == 0) {  // projection shortcut: downsample = bn(conv1x1_s(x)), module index li + 3
        if ((rc = conv_fwd(X, P(wts->w[li + 3]), wts->bias[li + 3], nullptr, D, B, h, w, cin, cout, 1, stride, 0, s))) return rc;
        shortcut = D;
      }
      if ((rc = conv_fwd(T2, P(wts->w[li + 2]), wts->bias[li + 2], shortcut, Y, B, ho, wo, planes, cout, 1, 1, 1, s))) return rc;
      std::swap(X, Y);
      li += blk == 0 ? 4 : 3;
      cin = cout; h = ho; w = wo;
    }
  }
  return global_avgpool(X, feat_out, B, h * w, cin, s);
}
