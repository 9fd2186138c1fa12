// K1 / K3 / K5: 3x3 (pad 1) and 1x1 convolutions, stride 1 or 2, over NHWC bf16 activations as an
// implicit GEMM on the 5th-gen tensor cores (tcgen05.mma, fp32 accumulators in TMEM), operands
// staged by TMA.  One kernel covers
//   * conv fwd + bias + ReLU                      (reference: torchvision vgg19.features Conv2d+ReLU,
//                                                  called from models/vgg/vgg.py:87)
//   * conv dgrad (+ tap gradient, x ReLU mask)     (autograd of the above, pipelines.py:90) -- a 3x3
//                                                  conv of dY with the 180-degree-rotated, transposed filter
//   * Gram backward dF = F . D_b (1x1, per-image D) (autograd of utils.py:253-256)
//
// GEMM view: M = pixels (a TW x TH x TB patch = 128 rows per M-tile, MT M-tiles per CTA),
// N = Cout tile (BN), K = ntaps * Cin walked as (tap, 64-channel chunk).  For every K block the
// producer issues one 4-D TMA box load per M-tile at the tap-shifted coordinate (out-of-bounds
// rows/cols are zero-filled by TMA == the conv's zero padding) and one 2-D load of the weight slab.
// Stride 2 (ResNet-50 bottlenecks, torchvision resnet50 via models/gaze_estimators/gaze_estimators.py:180-223): the
// activation map traverses W and H with element stride 2, so a 2TW x 2TH box starting at (2 x0 + kx - 1, 2 y0 + ky - 1)
// lands the TW x TH input pixels of the output patch in the same swizzled tile.
// The A/B tiles land in the SWIZZLE_128B K-major layout tcgen05 consumes directly.
//
// Warp roles (192 threads): warp 0 = TMA producer, warp 1 = TMEM allocator + MMA issuer,
// warps 2..5 = epilogue (TMEM -> registers -> bias/ReLU/mask/tap-gradient -> bf16 -> swizzled smem ->
// TMA store).
#include "isx_common.cuh"
#include "isx_internal.h"
#include "isx_kernels.h"

namespace isx {

struct ConvParams {
  int B, H, W, Cin, Cout;    // H, W: OUTPUT size (the input is stride x larger, rounded up)
  int ntaps;                 // 9 or 1
  int stride;                // 1 or 2
  int TW, TH, TB;            // patch shape, TW*TH*TB == 128
  int tiles_x, tiles_y, tiles_b;
  int n_tiles;               // Cout / BN
  int w_rows_per_image;      // 0, or Cout when every image has its own [Cout x Cin] matrix (Gram bwd)
  int extra_kb;              // fused Gram backward: extra K blocks (C/64) of  act(centre tap) x D_b  after the taps
  int stages;
  int relu;
  const float* bias;         // [Cout] or null
  const __nv_bfloat16* mask_act;  // [B,H,W,Cout] or null: out = act > 0 ? out : 0
  const __nv_bfloat16* add_buf;   // [B,H,W,Cout] or null: out += add
  const float* aff_a;        // [B,Cout] or null: out += aff_a + aff_b * act   (BN-statistics tap gradient)
  const float* aff_b;
  int fuse_pool;             // epilogue also emits the 2x2 max-pooled tile (TW, TH even) through tmP
  uint8_t* pool_idx;         // with fuse_pool: routing bytes of the max-pool + ReLU backward [B,H/2,W/2,Cout] or null
  int skip_out;              // with fuse_pool + pool_idx: the full-resolution tile is not stored
  // EPI == 1 (image-gradient tail, BN = 16): dx fp32 NCHW [B,xc,H,W] = acc[c] * mask / std[c]
  float* dx_nchw;
  int xc;
  const float* in_mask;      // [mask_b,1,H,W] or null
  int mask_b;
};

static constexpr int kATileBytes = 128 * 128;  // 128 rows x 64 bf16

static constexpr int kConvThreads = 64 + 256;  // TMA warp, MMA warp, 8 epilogue warps (two per TMEM lane quadrant)

template <int BN, int MT, int EPI>
__global__ void __launch_bounds__(kConvThreads, 2)
conv_tc_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
               const __grid_constant__ CUtensorMap tmO, const __grid_constant__ CUtensorMap tmM,
               const __grid_constant__ CUtensorMap tmA2, const __grid_constant__ CUtensorMap tmB2,
               const __grid_constant__ CUtensorMap tmP, const ConvParams p) {
  constexpr int kBTileBytes = BN * 128;
  constexpr int kStageBytes = MT * kATileBytes + kBTileBytes;
  constexpr int kTmemCols = (MT * BN) <= 32 ? 32 : (MT * BN) <= 64 ? 64 : (MT * BN) <= 128 ? 128 : (MT * BN) <= 256 ? 256 : 512;
  static_assert(MT * BN <= 512, "accumulators exceed TMEM");

  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const int stages = p.stages;
  const int ring_bytes = stages * kStageBytes;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + ring_bytes);
  uint64_t* empty_bar = full_bar + stages;
  uint64_t* tmem_full_bar = empty_bar + stages;
  uint64_t* epi_bar = tmem_full_bar + 1;  // [2]: TMA loads of the ReLU-mask activation tile for the epilogue
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(epi_bar + 2);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  // ---- tile coordinates --------------------------------------------------------------------
  const int n_tile = blockIdx.x % p.n_tiles;
  const int sp_super = blockIdx.x / p.n_tiles;
  const int n0 = n_tile * BN;
  int x0[MT], y0[MT], b0[MT];
#pragma unroll
  for (int mt = 0; mt < MT; ++mt) {
    int t = sp_super * MT + mt;
    int tx = t % p.tiles_x;
    int r = t / p.tiles_x;
    int ty = r % p.tiles_y;
    int tb = r / p.tiles_y;  // may exceed tiles_b for the padded last super-tile: fully out of bounds
    x0[mt] = tx * p.TW;
    y0[mt] = ty * p.TH;
    b0[mt] = tb * p.TB;
  }

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    if (EPI == 0) tma_prefetch_desc(&tmO);
    if (EPI == 0 && p.mask_act != nullptr) tma_prefetch_desc(&tmM);
    if (p.extra_kb > 0) { tma_prefetch_desc(&tmA2); tma_prefetch_desc(&tmB2); }
    if (p.fuse_pool) tma_prefetch_desc(&tmP);
    for (int s = 0; s < stages; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    mbar_init(tmem_full_bar, 1);
    mbar_init(&epi_bar[0], 1);
    mbar_init(&epi_bar[1], 1);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc<kTmemCols>(tmem_ptr_smem);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;

  const int cin_blocks = p.Cin >> 6;
  const int num_kb_conv = p.ntaps * cin_blocks;
  const int num_kb = num_kb_conv + p.extra_kb;

  if (warp == 0) {
    // ================================ TMA producer =========================================
    if (lane == 0) {
      const int wrow0 = (p.w_rows_per_image ? b0[0] * p.w_rows_per_image : 0) + n0;
      const int stride = EPI == 0 ? p.stride : 1;  // the image-gradient tail is stride 1
      // running stage / tap / channel-block counters (no division on the producer's critical path)
      int s = 0, tap = 0, cb = 0, ky = p.ntaps == 9 ? 0 : 1, kx = p.ntaps == 9 ? 0 : 1;
      uint32_t ph = 0;
      for (int kb = 0; kb < num_kb; ++kb) {
        const int sb = s;
        mbar_wait(&empty_bar[sb], ph ^ 1);
        mbar_arrive_expect_tx(&full_bar[sb], kStageBytes);
        uint8_t* st = smem + sb * kStageBytes;
        if (++s == stages) { s = 0; ph ^= 1; }
        if (kb < num_kb_conv) {
#pragma unroll
          for (int mt = 0; mt < MT; ++mt)
            tma_load_4d(st + mt * kATileBytes, &tmA, &full_bar[sb], cb * 64, x0[mt] * stride + kx - 1,
                        y0[mt] * stride + ky - 1, b0[mt]);
          tma_load_2d(st + MT * kATileBytes, &tmB, &full_bar[sb], cb * 64, tap * p.Cout + wrow0);
          if (++cb == cin_blocks) {
            cb = 0; ++tap;
            if (p.ntaps == 9 && ++kx == 3) { kx = 0; ++ky; }
          }
        } else {
          // fused Gram backward: dX += F . D_b  (F = activation of the layer below, D_b = dL/dG of image b)
          const int cb2 = kb - num_kb_conv;
#pragma unroll
          for (int mt = 0; mt < MT; ++mt)
            tma_load_4d(st + mt * kATileBytes, &tmA2, &full_bar[sb], cb2 * 64, x0[mt], y0[mt], b0[mt]);
          tma_load_2d(st + MT * kATileBytes, &tmB2, &full_bar[sb], cb2 * 64, b0[0] * p.Cout + n0);
        }
      }
    }
  } else if (warp == 1) {
    // ================================ MMA issuer ===========================================
    if (lane == 0) {
      constexpr uint32_t idesc = umma_idesc_bf16(128, BN, false, false);
      // The issuing thread is the bottleneck of the N <= 128 tiles (isx_common.cuh, umma_bf16_lohi): one descriptor is
      // built here, every MMA adds an immediate to its low word.
      const uint64_t d0 = umma_desc_sw128(smem_u32(smem), 16, 1024);
      const uint32_t d_hi = static_cast<uint32_t>(d0 >> 32);
      uint32_t a_lo = static_cast<uint32_t>(d0);
      int s = 0;
      uint32_t ph = 0;
      // An mbarrier probe costs ~150 cycles even when its phase completed long ago; the probe of the NEXT stage is issued
      // before this stage's MMAs and consumed after them (profiles/r01_umma_issue_probe.txt).
      bool ready = false;
      for (int kb = 0; kb < num_kb; ++kb) {
        if (!ready) mbar_wait(&full_bar[s], ph);
        tc_fence_after();
        const uint32_t a_cur = a_lo;
        const int s_cur = s;
        a_lo += kStageBytes >> 4;
        if (++s == stages) { s = 0; ph ^= 1; a_lo = static_cast<uint32_t>(d0); }
        ready = (kb + 1 < num_kb) && mbar_try_wait(&full_bar[s], ph);
#pragma unroll
        for (int mt = 0; mt < MT; ++mt) {
#pragma unroll
          for (int k = 0; k < 4; ++k)  // 4 x UMMA_K(16) = 64 channels
            umma_bf16_lohi(tmem_base + mt * BN, a_cur + ((mt * kATileBytes + k * 32) >> 4), d_hi,
                           a_cur + ((MT * kATileBytes + k * 32) >> 4), d_hi, idesc, (kb | k) != 0 ? 1u : 0u);
        }
        umma_commit(&empty_bar[s_cur]);  // frees the smem stage once these MMAs have read it
      }
      umma_commit(tmem_full_bar);
    }
  } else if (warp >= 2) {
    // ================================ epilogue =============================================
    const int q = warp & 3;  // TMEM lane quadrant this warp may access
    const int hsel = (warp - 2) >> 2;  // which 32-column half of every 64-channel group this warp converts
    const int row = q * 32 + lane;
    mbar_wait(tmem_full_bar, 0);
    tc_fence_after();
    const int tw = row % p.TW;
    const int th = (row / p.TW) % p.TH;
    const int tb = row / (p.TW * p.TH);
    if constexpr (EPI == 1) {
      // image-gradient tail: 3 (of 16) accumulator columns -> fp32 NCHW planes, Normalize backward (1/std), mask
#pragma unroll 1
      for (int mt = hsel == 0 ? 0 : MT; mt < MT; ++mt) {
        const int x = x0[mt] + tw, y = y0[mt] + th, b = b0[mt] + tb;
        const bool valid = (x < p.W) && (y < p.H) && (b < p.B);
        uint32_t v[16];
        tmem_ld_32x16(tmem_base + (static_cast<uint32_t>(q * 32) << 16) + mt * BN, v);
        tmem_ld_wait();
        if (valid) {
          const size_t hw = static_cast<size_t>(p.H) * p.W;
          const size_t off = static_cast<size_t>(y) * p.W + x;
          float m = 1.f;
          if (p.in_mask != nullptr) m = __ldg(p.in_mask + (p.mask_b > 1 ? b : 0) * hw + off);
          const float a0 = __uint_as_float(v[0]) * m / 0.229f;
          const float a1 = __uint_as_float(v[1]) * m / 0.224f;
          const float a2 = __uint_as_float(v[2]) * m / 0.225f;
          if (p.xc == 3) {
            float* o = p.dx_nchw + static_cast<size_t>(b) * 3 * hw + off;
            o[0] = a0; o[hw] = a1; o[2 * hw] = a2;
          } else {
            p.dx_nchw[static_cast<size_t>(b) * hw + off] = a0 + a1 + a2;
          }
        }
      }
    } else {
    constexpr int NG = MT * (BN / 64);                 // 64-channel output groups of this CTA
    uint8_t* scratch = smem + NG * kATileBytes;          // 2 x 16 KB: ReLU-mask activation tiles (TMA, swizzled)
    const bool use_mask = p.mask_act != nullptr;
    auto issue_mask_load = [&](int gi) {
      const int mt_ = gi / (BN / 64), g_ = gi % (BN / 64);
      mbar_arrive_expect_tx(&epi_bar[gi & 1], kATileBytes);
      tma_load_4d(scratch + (gi & 1) * kATileBytes, &tmM, &epi_bar[gi & 1], n0 + g_ * 64, x0[mt_], y0[mt_], b0[mt_]);
    };
    if (use_mask && threadIdx.x == 64) {
      issue_mask_load(0);
      if (NG > 1) issue_mask_load(1);
    }
#pragma unroll 1
    for (int mt = 0; mt < MT; ++mt) {
      const int x = x0[mt] + tw, y = y0[mt] + th, b = b0[mt] + tb;
      const bool valid = (x < p.W) && (y < p.H) && (b < p.B);
      const size_t pix = valid ? ((static_cast<size_t>(b) * p.H + y) * p.W + x) * p.Cout : 0;
#pragma unroll 1
      for (int g = 0; g < BN / 64; ++g) {
        const int gi = mt * (BN / 64) + g;
        uint8_t* stg = smem + gi * kATileBytes;  // pipeline smem is drained by now
        const uint8_t* mrow = scratch + (gi & 1) * kATileBytes + row * 128;
        if (use_mask) mbar_wait(&epi_bar[gi & 1], (gi >> 1) & 1);
        {
          const int h = hsel;
          const int nloc = g * 64 + h * 32;
          uint32_t v[32];
          tmem_ld_32x32(tmem_base + (static_cast<uint32_t>(q * 32) << 16) + mt * BN + nloc, v);
          tmem_ld_wait();
          float f[32];
#pragma unroll
          for (int i = 0; i < 32; ++i) f[i] = __uint_as_float(v[i]);
          const int n = n0 + nloc;
          if (p.bias != nullptr) {
#pragma unroll
            for (int i = 0; i < 32; i += 4) {
              const float4 bv = __ldg(reinterpret_cast<const float4*>(p.bias + n + i));
              f[i] += bv.x; f[i + 1] += bv.y; f[i + 2] += bv.z; f[i + 3] += bv.w;
            }
          }
          if (p.add_buf != nullptr && valid) {
#pragma unroll
            for (int i = 0; i < 32; i += 8) {
              const uint4 u = __ldg(reinterpret_cast<const uint4*>(p.add_buf + pix + n + i));
              float2 t;
              t = unpack_bf16x2(u.x); f[i] += t.x; f[i + 1] += t.y;
              t = unpack_bf16x2(u.y); f[i + 2] += t.x; f[i + 3] += t.y;
              t = unpack_bf16x2(u.z); f[i + 4] += t.x; f[i + 5] += t.y;
              t = unpack_bf16x2(u.w); f[i + 6] += t.x; f[i + 7] += t.y;
            }
          }
          if (use_mask) {
            // out-of-bounds rows of the box were zero-filled by TMA: act = 0 -> gradient 0 (never stored anyway)
#pragma unroll
            for (int i = 0; i < 32; i += 8) {
              const int chunk = (h * 4 + (i >> 3)) ^ (row & 7);
              const uint4 u = *reinterpret_cast<const uint4*>(mrow + chunk * 16);
              float a[8];
              float2 t;
              t = unpack_bf16x2(u.x); a[0] = t.x; a[1] = t.y;
              t = unpack_bf16x2(u.y); a[2] = t.x; a[3] = t.y;
              t = unpack_bf16x2(u.z); a[4] = t.x; a[5] = t.y;
              t = unpack_bf16x2(u.w); a[6] = t.x; a[7] = t.y;
              if (p.aff_a != nullptr && valid) {
                const float* pa = p.aff_a + static_cast<size_t>(b) * p.Cout + n + i;
                const float* pb = p.aff_b + static_cast<size_t>(b) * p.Cout + n + i;
#pragma unroll
                for (int j = 0; j < 8; ++j) f[i + j] += __ldg(pa + j) + __ldg(pb + j) * a[j];
              }
#pragma unroll
              for (int j = 0; j < 8; ++j) f[i + j] = a[j] > 0.f ? f[i + j] : 0.f;
            }
          }
          if (p.relu) {
#pragma unroll
            for (int i = 0; i < 32; ++i) f[i] = fmaxf(f[i], 0.f);
          }
          // 32 channels -> 4 x 16 B chunks of this row, 128B-swizzled like the TMA box layout
          uint8_t* rowp = stg + row * 128;
#pragma unroll
          for (int c = 0; c < 4; ++c) {
            uint4 o;
            o.x = pack_bf16x2(f[c * 8 + 0], f[c * 8 + 1]);
            o.y = pack_bf16x2(f[c * 8 + 2], f[c * 8 + 3]);
            o.z = pack_bf16x2(f[c * 8 + 4], f[c * 8 + 5]);
            o.w = pack_bf16x2(f[c * 8 + 6], f[c * 8 + 7]);
            const int chunk = (h * 4 + c) ^ (row & 7);
            *reinterpret_cast<uint4*>(rowp + chunk * 16) = o;
          }
        }
        fence_proxy_async_smem();
        asm volatile("bar.sync 1, 256;" ::: "memory");  // the eight epilogue warps
        if (threadIdx.x == 64) {
          if (!p.skip_out) {
            tma_store_4d(&tmO, stg, n0 + g * 64, x0[mt], y0[mt], b0[mt]);
            tma_store_commit();
          }
          if (use_mask && gi + 2 < NG) issue_mask_load(gi + 2);  // scratch slot (gi & 1) has been read by everyone
        }
        if (p.fuse_pool) {
          // K2 fused: 2x2 max-pool of the staged bf16 tile -> 32 pooled pixels x 64 channels (MaxPool2d(2,2) after ReLU)
          uint8_t* pst = smem + (NG + (use_mask ? 2 : 0)) * kATileBytes + gi * 4096;
          const int twp = p.TW >> 1, thp = p.TH >> 1;
          const int et = threadIdx.x - 64;  // 0..255
          {
            const int item = et;
            const int pr = item >> 3, chunk = item & 7;
            const int px = pr % twp, py = (pr / twp) % thp, pb = pr / (twp * thp);
            const int r00 = (pb * p.TH + 2 * py) * p.TW + 2 * px;
            const int rr[4] = {r00, r00 + 1, r00 + p.TW, r00 + p.TW + 1};
            uint4 u4[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) u4[k] = *reinterpret_cast<const uint4*>(stg + rr[k] * 128 + ((chunk ^ (rr[k] & 7)) * 16));
            uint4 m4;
            uint2 codes;
            pool4_codes(u4, m4, codes);
            if (p.pool_idx != nullptr) {  // routing bytes of the max-pool + ReLU backward, straight to global memory
              const int xp = (x0[mt] >> 1) + px, yp = (y0[mt] >> 1) + py, bp = b0[mt] + pb;
              if (xp < (p.W >> 1) && yp < (p.H >> 1) && bp < p.B)
                *reinterpret_cast<uint2*>(p.pool_idx + ((static_cast<size_t>(bp) * (p.H >> 1) + yp) * (p.W >> 1) + xp) * p.Cout +
                                          n0 + g * 64 + chunk * 8) = codes;
            }
            *reinterpret_cast<uint4*>(pst + pr * 128 + ((chunk ^ (pr & 7)) * 16)) = m4;
          }
          fence_proxy_async_smem();
          asm volatile("bar.sync 1, 256;" ::: "memory");
          if (threadIdx.x == 64) {
            tma_store_4d(&tmP, pst, n0 + g * 64, x0[mt] >> 1, y0[mt] >> 1, b0[mt]);
            tma_store_commit();
          }
        }
      }
    }
    }
    if (EPI == 0 && threadIdx.x == 64) tma_store_wait_all<0>();
    tc_fence_before();
  }
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc<kTmemCols>(tmem_base);
  }
}

// Pick the 128-pixel patch shape (TW x TH x TB) with the least padding; ties -> wider rows.
static void choose_patch(int B, int H, int W, bool one_image_per_tile, int* TW, int* TH, int* TB) {
  long best = -1;
  for (int tw = 128; tw >= 1; tw >>= 1) {
    for (int th = 128 / tw; th >= 1; th >>= 1) {
      int tb = 128 / (tw * th);
      if (one_image_per_tile && tb != 1) continue;
      if (tw > 256 || th > 256 || tb > 256) continue;
      long padded = static_cast<long>((W + tw - 1) / tw * tw) * ((H + th - 1) / th * th) * ((B + tb - 1) / tb * tb);
      if (best < 0 || padded < best) {
        best = padded;
        *TW = tw; *TH = th; *TB = tb;
      }
    }
  }
}

template <int BN, int MT, int EPI = 0>
static int launch_conv(const ConvArgs& a, int stages_override, cudaStream_t stream) {
  ConvParams p;
  memset(&p, 0, sizeof(p));
  const int Ho = (a.H + a.stride - 1) / a.stride, Wo = (a.W + a.stride - 1) / a.stride;  // output size
  p.B = a.B; p.H = Ho; p.W = Wo; p.Cin = a.Cin; p.Cout = a.Cout; p.ntaps = a.ntaps; p.stride = a.stride;
  const bool per_image = a.per_image_weights || a.gram_act != nullptr;
  choose_patch(a.B, Ho, Wo, per_image, &p.TW, &p.TH, &p.TB);
  p.tiles_x = (Wo + p.TW - 1) / p.TW;
  p.tiles_y = (Ho + p.TH - 1) / p.TH;
  p.tiles_b = (a.B + p.TB - 1) / p.TB;
  p.n_tiles = a.Cout / BN;
  p.w_rows_per_image = a.per_image_weights ? a.Cout : 0;
  p.relu = a.relu; p.bias = a.bias; p.mask_act = a.mask_act; p.add_buf = a.add_buf;
  p.aff_a = a.aff_a; p.aff_b = a.aff_b;
  p.dx_nchw = a.dx_nchw; p.xc = a.xc; p.in_mask = a.in_mask; p.mask_b = a.mask_b;
  p.extra_kb = a.gram_act != nullptr ? a.Cout / 64 : 0;
  if (per_image && MT != 1)  // both M-tiles of a CTA must lie in one image (they share the per-image B slab)
    ISX_REQUIRE(p.TB == 1 && (p.tiles_x * p.tiles_y) % MT == 0, "per-image weights: an odd tile count per image needs MT = 1");

  constexpr int kStageBytes = MT * kATileBytes + BN * 128;
  // epilogue staging (one 16 KB tile per 64-channel group) + 2 mask-tile slots alias the drained pipeline
  const bool fuse_pool = EPI == 0 && a.pool_out != nullptr && p.TW % 2 == 0 && p.TH % 2 == 0 &&
                         a.H >= 2 && a.W >= 2;
  p.fuse_pool = fuse_pool ? 1 : 0;
  p.pool_idx = fuse_pool ? a.pool_idx : nullptr;
  p.skip_out = (fuse_pool && a.pool_idx != nullptr && a.skip_out) ? 1 : 0;
  const int epi_bytes = (MT * (BN / 64) + (a.mask_act ? 2 : 0)) * kATileBytes + (fuse_pool ? MT * (BN / 64) * 4096 : 0);
  int stages;
  size_t ring_bytes;
  stages = stages_override > 0 ? stages_override : (200 * 1024) / kStageBytes;
  if (stages > 8) stages = 8;
  if (stages < 2) stages = 2;
  while (stages * kStageBytes < epi_bytes) ++stages;
  ring_bytes = static_cast<size_t>(stages) * kStageBytes;
  p.stages = stages;
  const size_t smem_bytes = 1024 + ring_bytes + 256;
  ISX_REQUIRE(smem_bytes <= 227 * 1024, "conv_tc: %zu B of shared memory exceed 227 KB", smem_bytes);

  CUtensorMap tmA, tmB, tmO, tmM, tmA2, tmB2, tmP;
  {
    uint64_t dims[4] = {(uint64_t)a.Cin, (uint64_t)a.W, (uint64_t)a.H, (uint64_t)a.B};
    uint64_t str[3] = {(uint64_t)a.Cin * 2, (uint64_t)a.W * a.Cin * 2, (uint64_t)a.H * a.W * a.Cin * 2};
    uint32_t box[4] = {64, (uint32_t)(p.TW * a.stride), (uint32_t)(p.TH * a.stride), (uint32_t)p.TB};
    const uint32_t es[4] = {1, (uint32_t)a.stride, (uint32_t)a.stride, 1};
    if (isx_make_tmap_bf16(&tmA, a.in, 4, dims, str, box, true, es)) return 3;
  }
  {
    uint64_t rows = (uint64_t)a.ntaps * a.Cout * (a.per_image_weights ? a.B : 1);
    uint64_t dims[2] = {(uint64_t)a.Cin, rows};
    uint64_t str[1] = {(uint64_t)a.Cin * 2};
    uint32_t box[2] = {64, (uint32_t)BN};
    if (isx_make_tmap_bf16(&tmB, a.weight, 2, dims, str, box, true)) return 3;
  }
  if (EPI == 0) {
    uint64_t dims[4] = {(uint64_t)a.Cout, (uint64_t)Wo, (uint64_t)Ho, (uint64_t)a.B};
    uint64_t str[3] = {(uint64_t)a.Cout * 2, (uint64_t)Wo * a.Cout * 2, (uint64_t)Ho * Wo * a.Cout * 2};
    uint32_t box[4] = {64, (uint32_t)p.TW, (uint32_t)p.TH, (uint32_t)p.TB};
    if (isx_make_tmap_bf16(&tmO, a.out, 4, dims, str, box, true)) return 3;
  } else {
    tmO = tmA;  // unused by the image-gradient epilogue
  }
  tmM = tmO; tmA2 = tmA; tmB2 = tmB; tmP = tmO;
  if (fuse_pool) {
    uint64_t dims[4] = {(uint64_t)a.Cout, (uint64_t)(a.W / 2), (uint64_t)(a.H / 2), (uint64_t)a.B};
    uint64_t str[3] = {(uint64_t)a.Cout * 2, (uint64_t)(a.W / 2) * a.Cout * 2, (uint64_t)(a.H / 2) * (a.W / 2) * a.Cout * 2};
    uint32_t box[4] = {64, (uint32_t)(p.TW / 2), (uint32_t)(p.TH / 2), (uint32_t)p.TB};
    if (isx_make_tmap_bf16(&tmP, a.pool_out, 4, dims, str, box, true)) return 3;
  }
  if (EPI == 0 && a.mask_act != nullptr) {
    uint64_t dims[4] = {(uint64_t)a.Cout, (uint64_t)a.W, (uint64_t)a.H, (uint64_t)a.B};
    uint64_t str[3] = {(uint64_t)a.Cout * 2, (uint64_t)a.W * a.Cout * 2, (uint64_t)a.H * a.W * a.Cout * 2};
    uint32_t box[4] = {64, (uint32_t)p.TW, (uint32_t)p.TH, (uint32_t)p.TB};
    if (isx_make_tmap_bf16(&tmM, a.mask_act, 4, dims, str, box, true)) return 3;
  }
  if (a.gram_act != nullptr) {  // K = Cout channels of the layer below (its activation is [B,H,W,Cout] too)
    uint64_t dims[4] = {(uint64_t)a.Cout, (uint64_t)a.W, (uint64_t)a.H, (uint64_t)a.B};
    uint64_t str[3] = {(uint64_t)a.Cout * 2, (uint64_t)a.W * a.Cout * 2, (uint64_t)a.H * a.W * a.Cout * 2};
    uint32_t box[4] = {64, (uint32_t)p.TW, (uint32_t)p.TH, (uint32_t)p.TB};
    if (isx_make_tmap_bf16(&tmA2, a.gram_act, 4, dims, str, box, true)) return 3;
    uint64_t dims2[2] = {(uint64_t)a.Cout, (uint64_t)a.Cout * a.B};
    uint64_t str2[1] = {(uint64_t)a.Cout * 2};
    uint32_t box2[2] = {64, (uint32_t)BN};
    if (isx_make_tmap_bf16(&tmB2, a.gram_D, 2, dims2, str2, box2, true)) return 3;
  }
  const long sp_tiles = static_cast<long>(p.tiles_x) * p.tiles_y * p.tiles_b;
  long grid = ((sp_tiles + MT - 1) / MT) * p.n_tiles;
  auto kern = conv_tc_kernel<BN, MT, EPI>;
  ISX_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bytes));
  isx_prof_begin(ISX_PROF_CONV,
                 2.0 * (a.ntaps * a.Cin + (a.gram_act ? a.Cout : 0)) * a.Cout * static_cast<double>(a.B) * Ho * Wo, stream);
  kern<<<(unsigned)grid, kConvThreads, smem_bytes, stream>>>(tmA, tmB, tmO, tmM, tmA2, tmB2, tmP, p);
  isx_prof_end(ISX_PROF_CONV, stream);
  ISX_LAUNCH_CHECK();
  if (a.pool_out != nullptr && !fuse_pool) {  // patch shape not poolable in the epilogue: separate kernel
    if (a.pool_idx != nullptr) return maxpool_fwd_idx(a.out, a.pool_out, a.pool_idx, a.B, a.H, a.W, a.Cout, stream);
    return maxpool_fwd(a.out, a.pool_out, a.B, a.H, a.W, a.Cout, stream);
  }
  return 0;
}

int conv_tc(const ConvArgs& a_in, cudaStream_t stream) {
  ConvArgs a = a_in;
  ISX_REQUIRE(a.stride == 1 || (a.stride == 2 && a.pool_out == nullptr && a.mask_act == nullptr && a.gram_act == nullptr &&
                                a.dx_nchw == nullptr && !a.per_image_weights),
              "conv_tc: stride %d (stride 2 is the plain forward conv: no pool, mask, image gradient or per-image weights)",
              a.stride);
  if (a.dx_nchw != nullptr && isx_ctx()->opt_tail_n > 0 && isx_ctx()->opt_c64 < 2 && a.force_bn == 0 &&
      a.Cin == 64 && a.Cout == 16 && a.ntaps == 9)
    return conv1_1_tail_n(a.in, a.weight, a.in_mask, a.mask_b, a.dx_nchw, a.xc, a.B, a.H, a.W, stream);
  if (isx_ctx()->opt_sweep64 > 0 && a.force_bn == 0 && !a.generic_only && conv_sweep_applicable(a)) {
    // strips of 128 pixels along the better-fitting image axis, every CTA sweeps an equal share of them: worth it when the
    // strips are mostly real pixels (the kernel is ~1.5x faster per processed pixel than conv_c64) and every SM gets a few
    // hundred of them (a CTA's share starts and ends with two slower edge strips)
    const long strips = static_cast<long>(a.B) * ((std::max(a.H, a.W) + 127) / 128) * std::min(a.H, a.W);
    // measured (profiles/r02_conv_sweep_experiment.txt), us per 640x400 image: forward 14.0-14.8 against 17.5-18.1 for conv_c64,
    // with the fused pool 15.7-17.4 against 18.6-19.7, dgrad + mask 19.9-20.1 against 21.5-22.0, dgrad + mask + Gram 21.9-22.2
    // against 23.5-25.6
    if (isx_ctx()->opt_sweep64 >= 2 ||
        (conv_sweep_efficiency(a) >= 0.85 && strips >= 64L * kNumSMs && std::min(a.H, a.W) >= 16))
      return conv_sweep(a, stream);
  }
  if (isx_ctx()->opt_c64 > 0 && a.force_bn == 0 && !a.generic_only && conv_c64_applicable(a) &&
      (isx_ctx()->opt_c64 >= 2 || (a.dx_nchw == nullptr && static_cast<long>(a.B) * ((a.H + 15) / 16) * ((a.W + 7) / 8) >= kNumSMs)))
    return conv_c64(a, stream);
  if (isx_ctx()->opt_halo2 > 0 && a.force_bn == 0 && !a.generic_only && conv_halo_applicable(a)) {
    const long items = static_cast<long>(a.B) * ((a.H + 15) / 16) * ((a.W + 15) / 16) * (a.Cout / (a.Cout % 128 == 0 ? 128 : 64));
    if (isx_ctx()->opt_halo2 >= 2 || (items >= 2 * kNumSMs && conv_halo_efficiency(a) >= 0.85)) return conv_halo(a, stream);
  }
  if (a.dx_nchw != nullptr) {  // conv1_1 dgrad tail: N = 16 (3 real output channels), fp32 NCHW epilogue
    ISX_REQUIRE(a.Cin == 64 && a.Cout == 16 && a.ntaps == 9, "conv_tc: image-gradient mode needs Cin 64, Cout 16 (padded)");
    ISX_REQUIRE(a.xc == 1 || a.xc == 3, "conv_tc: xc must be 1 or 3");
    const long pix_tiles = (static_cast<long>(a.B) * a.H * a.W + 127) / 128;
    if (a.force_mt == 1 || pix_tiles < 4 * kNumSMs) return launch_conv<16, 1, 1>(a, a.force_stages ? a.force_stages : 3, stream);
    return launch_conv<16, 2, 1>(a, a.force_stages ? a.force_stages : 2, stream);
  }
  ISX_REQUIRE(a.Cin % 64 == 0 && a.Cout % 64 == 0, "conv_tc: Cin=%d / Cout=%d must be multiples of 64", a.Cin, a.Cout);
  ISX_REQUIRE(a.ntaps == 9 || a.ntaps == 1, "conv_tc: ntaps must be 9 or 1");
  ISX_REQUIRE(a.B > 0 && a.H > 0 && a.W > 0, "conv_tc: empty input");
  ISX_REQUIRE((a.aff_a == nullptr) || (a.mask_act != nullptr), "conv_tc: affine tap gradient needs the activation");
  ISX_REQUIRE((a.gram_act == nullptr) || (a.gram_D != nullptr && !a.per_image_weights), "conv_tc: bad fused-Gram arguments");
  int bn = a.force_bn, mt = a.force_mt;
  int st = a.force_stages;
  if (bn == 0) {
    // Measured on B200 (profiles/r01_conv_tile_sweep.txt): two pipeline stages and >= 2 co-resident CTAs per SM
    // (one CTA's epilogue overlaps the other's main loop) beat deeper pipelines with one CTA per SM.
    //   Cout  64: BN  64, two M-tiles per CTA (the weight slab is shared by 256 pixels)
    //   Cout 128: BN 128, two M-tiles
    //   Cout 256+: BN 256, one M-tile
    bn = a.Cout % 256 == 0 ? 256 : (a.Cout % 128 == 0 ? 128 : 64);
    mt = (bn == 256 || a.per_image_weights) ? 1 : 2;
    if (st == 0) st = 2;
    // small problems: prefer more CTAs over bigger tiles
    const long pix_tiles = (static_cast<long>(a.B) * ((a.H + a.stride - 1) / a.stride) * ((a.W + a.stride - 1) / a.stride) + 127) / 128;
    auto ctas = [&](int BN_, int MT_) { return ((pix_tiles + MT_ - 1) / MT_) * (a.Cout / BN_); };
    if (ctas(bn, mt) < 2 * kNumSMs && mt == 2) mt = 1;
    if (ctas(bn, mt) < 2 * kNumSMs && bn == 256) bn = 128;
    if (a.gram_act != nullptr && mt == 2) {  // fused Gram backward: both M-tiles must share one image
      int tw, th, tb;
      choose_patch(a.B, a.H, a.W, true, &tw, &th, &tb);
      if ((((a.W + tw - 1) / tw) * ((a.H + th - 1) / th)) % 2 != 0) mt = 1;
    }
  }
  if (mt == 0) mt = 1;
#define ISX_CONV_CASE(BN_, MT_) \
  if (bn == BN_ && mt == MT_) return launch_conv<BN_, MT_>(a, st, stream);
  ISX_CONV_CASE(64, 1) ISX_CONV_CASE(64, 2) ISX_CONV_CASE(128, 1) ISX_CONV_CASE(128, 2)
  ISX_CONV_CASE(256, 1) ISX_CONV_CASE(256, 2)
#undef ISX_CONV_CASE
  ISX_REQUIRE(false, "conv_tc: unsupported tile BN=%d MT=%d", bn, mt);
}

}  // namespace isx
