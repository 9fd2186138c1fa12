// K0 + K1 head on the tensor cores: Normalize -> [* mask] -> conv1_1 (3 -> 64, K = 27) + bias + ReLU
// (models/vgg/vgg.py:81-87).  The 27-tap patch of every pixel is gathered by the pixel's own thread from the
// fp32 NCHW image: a CTA first normalises the (TH+2) x (TW+2) x 3 input patch of its TW x TH pixel tile ONCE
// into shared memory as (bf16 hi, bf16 lo) word pairs (16 mantissa bits survive), then every thread copies
// the 27 words of its pixel into one 128-byte K-major row [hi0 lo0 hi1 lo1 ... | 0] of the A tile in tcgen05's
// SWIZZLE_128B layout; the weight slab [64][w0 w0 w1 w1 ... | 0] is loaded once per CTA by TMA.  One 128x64x64 MMA per 128 pixels, fp32
// accumulation in TMEM, bias + ReLU + bf16 in the epilogue, TMA store of the NHWC rows.
#include <algorithm>

#include "isx_common.cuh"
#include "isx_kernels.h"

namespace isx {

__global__ void pack_w0_fwd_kernel(const float* __restrict__ w, __nv_bfloat16* __restrict__ wp) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;  // [64][64]
  if (i >= 64 * 64) return;
  const int k = i % 64, o = i / 64;
  const float v = k < 54 ? w[o * 27 + (k >> 1)] : 0.f;  // K index 2j (x hi_j) and 2j+1 (x lo_j) share w_j
  wp[i] = __float2bfloat16_rn(v);
}

int pack_w0_fwd(const float* w, __nv_bfloat16* wp, cudaStream_t s) {
  pack_w0_fwd_kernel<<<16, 256, 0, s>>>(w, wp);
  ISX_LAUNCH_CHECK();
  return 0;
}

static constexpr int kC11Bias = 16384 + 8192 + 64;   // shared-memory offsets behind the two operand tiles and the barriers
static constexpr int kC11Patch = kC11Bias + 256;

struct C11Params {
  const float* x;
  const float* mask;
  const float* bias;
  int xc, mask_b, B, H, W;
  int TW, TH, tiles_x, tiles_y;
  int n_tiles;
};


// TW (power of two, TH = 128 / TW) is a template parameter: the patch index arithmetic (i % PW, i / (PW*PH), tid % TW)
// then compiles to multiply-shift instead of ~15 integer divisions per thread and tile.
template <int TW>
__global__ void __launch_bounds__(128, 5)
conv1_1_tc_kernel(const __grid_constant__ CUtensorMap tmW, const __grid_constant__ CUtensorMap tmO, const C11Params p) {
  constexpr int TH = 128 / TW;
  // Everything lives in DYNAMIC shared memory declared 1024-byte aligned (no static arrays in front of it, no alignment
  // slack): 27 KB + the 1 KB the system reserves per CTA lets eight CTAs share an SM's 227 KB.
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* sA = smem;                 // 128 rows x 128 B
  uint8_t* sB = smem + 16384;         // 64 rows x 128 B
  uint8_t* sO = sA;                   // output staging aliases the A tile (free once the MMA has completed)
  uint64_t* w_bar = reinterpret_cast<uint64_t*>(smem + 16384 + 8192);
  uint64_t* mma_bar = w_bar + 1;
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(mma_bar + 1);
  float* s_bias = reinterpret_cast<float*>(smem + kC11Bias);
  uint32_t* s_patch = reinterpret_cast<uint32_t*>(smem + kC11Patch);   // 3 * (TW + 2) * (TH + 2) words
  const int tid = threadIdx.x, warp = tid >> 5;
  const float mean[3] = {0.485f, 0.456f, 0.406f};
  const float stdv[3] = {0.229f, 0.224f, 0.225f};

  if (tid == 0) {
    if (smem_u32(smem) & 1023u) {
      printf("isx: conv1_1 head: dynamic shared memory is not 1024-byte aligned\n");
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
    mbar_arrive_expect_tx(w_bar, 8192);
    tma_load_2d(sB, &tmW, w_bar, 0, 0);
  }
  const long hw = static_cast<long>(p.H) * p.W;
  constexpr uint32_t idesc = umma_idesc_bf16(128, 64, false, false);
  uint32_t phase = 0;
  bool w_ready = false;
  constexpr int PW = TW + 2, PH = TH + 2;
  constexpr int npatch = 3 * PH * PW;
  const int tw = tid % TW, th = tid / TW;
  // The raw patch values of the NEXT tile are fetched into registers before this tile's MMA + epilogue (their global /
  // L2 latency is the longest link of the per-tile chain) and normalised into shared memory at the top of the next round.
  constexpr int kMaxPerThread = (npatch + 127) / 128;  // patch words per thread
  float raw[kMaxPerThread], rawm[kMaxPerThread];
  auto fetch = [&](int tile) {
    const int tx = tile % p.tiles_x;
    const int ty = (tile / p.tiles_x) % p.tiles_y;
    const int b = tile / (p.tiles_x * p.tiles_y);
    const int x0 = tx * TW, y0 = ty * TH;
#pragma unroll
    for (int j = 0; j < kMaxPerThread; ++j) {
      const int i = tid + j * 128;
      raw[j] = 0.f; rawm[j] = 0.f;  // rawm = 0 marks zero padding of the NORMALISED image
      if (i < npatch) {
        const int px = i % PW;
        const int py = (i / PW) % PH;
        const int c = i / (PW * PH);
        const int y = y0 + py - 1, xq = x0 + px - 1;
        if (y >= 0 && y < p.H && xq >= 0 && xq < p.W) {
          const float* xp = p.x + (static_cast<long>(b) * p.xc + (p.xc == 3 ? c : 0)) * hw;
          raw[j] = __ldg(xp + static_cast<long>(y) * p.W + xq);
          rawm[j] = p.mask ? __ldg(p.mask + (static_cast<long>(p.mask_b > 1 ? b : 0) * p.H + y) * p.W + xq) : 1.f;
        }
      }
    }
  };
  if (static_cast<int>(blockIdx.x) < p.n_tiles) fetch(blockIdx.x);
  for (int tile = blockIdx.x; tile < p.n_tiles; tile += gridDim.x) {
    const int tx = tile % p.tiles_x;
    const int ty = (tile / p.tiles_x) % p.tiles_y;
    const int b = tile / (p.tiles_x * p.tiles_y);
    const int x0 = tx * TW, y0 = ty * TH;
    // ---- normalise + split the prefetched patch (zero padding applies to the NORMALISED image) ----
#pragma unroll
    for (int j = 0; j < kMaxPerThread; ++j) {
      const int i = tid + j * 128;
      if (i < npatch) {
        const int c = i / (PW * PH);
        // same expression as the oracle: ((x - mean) / std) * mask; padding stays exactly 0
        float t = (raw[j] - mean[c]) / stdv[c];
        t = rawm[j] == 0.f ? 0.f : (p.mask ? t * rawm[j] : t);
        const __nv_bfloat16 hi = __float2bfloat16_rn(t);
        const __nv_bfloat16 lo = __float2bfloat16_rn(t - __bfloat162float(hi));
        __nv_bfloat162 w2;
        w2.x = hi;
        w2.y = lo;
        s_patch[i] = *reinterpret_cast<uint32_t*>(&w2);
      }
    }
    if (tile + static_cast<int>(gridDim.x) < p.n_tiles) fetch(tile + gridDim.x);
    if (tid == 0) tma_store_wait_read<0>();  // previous tile's TMA store has finished reading sA (== staging)
    __syncthreads();
    // ---- this thread's pixel: 27 (hi, lo) words -> one swizzled 128-byte row ----
    uint32_t packed[32];
#pragma unroll
    for (int c = 0; c < 3; ++c)
#pragma unroll
      for (int ky = 0; ky < 3; ++ky)
#pragma unroll
        for (int kx = 0; kx < 3; ++kx) packed[c * 9 + ky * 3 + kx] = s_patch[(c * PH + th + ky) * PW + tw + kx];
#pragma unroll
    for (int k = 27; k < 32; ++k) packed[k] = 0u;
    uint8_t* rowp = sA + tid * 128;
#pragma unroll
    for (int c = 0; c < 8; ++c)
      *reinterpret_cast<uint4*>(rowp + ((c ^ (tid & 7)) * 16)) =
          make_uint4(packed[4 * c], packed[4 * c + 1], packed[4 * c + 2], packed[4 * c + 3]);
    fence_proxy_async_smem();  // generic-proxy smem writes -> visible to the tensor core (async proxy)
    __syncthreads();
    if (tid == 0) {
      if (!w_ready) mbar_wait(w_bar, 0);
      tc_fence_after();
      const uint32_t a_addr = smem_u32(sA), b_addr = smem_u32(sB);
#pragma unroll
      for (int k = 0; k < 4; ++k)
        umma_bf16(tmem_base, umma_desc_sw128(a_addr + k * 32, 16, 1024), umma_desc_sw128(b_addr + k * 32, 16, 1024),
                  idesc, k != 0 ? 1u : 0u);
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

int conv1_1_fwd_tc(const float* x, int xc, const float* mask, int mask_b, const __nv_bfloat16* w0_packed,
                   const float* bias, __nv_bfloat16* out, int B, int H, int W, cudaStream_t s) {
  ISX_REQUIRE(xc == 1 || xc == 3, "conv1_1: image must have 1 or 3 channels, got %d", xc);
  C11Params p;
  p.x = x; p.mask = mask; p.bias = bias; p.xc = xc; p.mask_b = mask_b; p.B = B; p.H = H; p.W = W;
  // 128-pixel tile TW x TH with the least work: padded pixels x the halo overhead of its (TW+2) x (TH+2) input patch
  // (16 x 8 reads 180 patch words per 128 pixels, 128 x 1 reads 390); ties go to the wider tile (coalesced image reads).
  double best = -1.0;
  for (int twc = 128; twc >= 1; twc >>= 1) {
    const int thc = 128 / twc;
    const double padded = static_cast<double>((W + twc - 1) / twc * twc) * ((H + thc - 1) / thc * thc);
    const double cost = padded * ((twc + 2) * (thc + 2));
    if (best < 0 || cost < best) { best = cost; p.TW = twc; p.TH = thc; }
  }
  p.tiles_x = (W + p.TW - 1) / p.TW;
  p.tiles_y = (H + p.TH - 1) / p.TH;
  const long nt = static_cast<long>(p.tiles_x) * p.tiles_y * B;
  ISX_REQUIRE(nt < (1L << 31), "conv1_1: too many tiles");
  p.n_tiles = static_cast<int>(nt);
  CUtensorMap tmW, tmO;
  {
    uint64_t dims[2] = {64, 64};
    uint64_t str[1] = {128};
    uint32_t box[2] = {64, 64};
    if (isx_make_tmap_bf16(&tmW, w0_packed, 2, dims, str, box, true)) return 3;
  }
  {
    uint64_t dims[4] = {64, (uint64_t)W, (uint64_t)H, (uint64_t)B};
    uint64_t str[3] = {128, (uint64_t)W * 128, (uint64_t)H * W * 128};
    uint32_t box[4] = {64, (uint32_t)p.TW, (uint32_t)p.TH, 1};
    if (isx_make_tmap_bf16(&tmO, out, 4, dims, str, box, true)) return 3;
  }
  const size_t smem_bytes = kC11Patch + 4 * 3 * (p.TW + 2) * (p.TH + 2);
  // Latency-bound kernel (per tile: patch -> smem, row build, MMA round trip, TMEM read, TMA store): what hides the chain
  // is the number of resident CTAs.  Compiled for five per SM (89-96 registers, 28 KB of shared memory and 64 TMEM columns
  // each).  A build for eight per SM (64 registers, 40-192 B of spill stores) was measured SLOWER on a B200: 12.7 against
  // 11.1 us/image at 640x400 -- the tile chain is bound by instruction issue and shared-memory traffic, not by occupancy.
  // Measured grid sweep at 640x400 (us/image, five resident): 148 x 5 12.0, x 6 15.4 (partial second wave), x 10 11.9,
  // x 32 11.8 -> many short CTAs make the static tile split insensitive to wave quantisation.
  const int grid = std::min(p.n_tiles, kNumSMs * 32);
#define ISX_C11_CASE(TW_)                                                                                                   \
  case TW_:                                                                                                                 \
    ISX_CHECK_CUDA(cudaFuncSetAttribute(conv1_1_tc_kernel<TW_>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bytes)); \
    conv1_1_tc_kernel<TW_><<<grid, 128, smem_bytes, s>>>(tmW, tmO, p);                                                      \
    break;
  switch (p.TW) {
    ISX_C11_CASE(128) ISX_C11_CASE(64) ISX_C11_CASE(32) ISX_C11_CASE(16) ISX_C11_CASE(8) ISX_C11_CASE(4) ISX_C11_CASE(2)
    ISX_C11_CASE(1)
    default: ISX_REQUIRE(false, "conv1_1: bad tile width %d", p.TW);
  }
#undef ISX_C11_CASE
  ISX_LAUNCH_CHECK();
  return 0;
}

}  // namespace isx
