// 3x3 convolutions with Cin = Cout = 64 (conv1_2 forward and dgrad; with option c64 = 2 also the 64 -> 3 image-gradient
// tail as an N = 16 tile, kept for tests -- the default tail is conv1_1_tail.cu).  In the generic kernel these layers
// re-load a 16 KB A tile and an 8 KB weight slab for every tap; here:
//   * the nine weight slabs (9 x BN x 64 bf16 = 72 KB for BN = 64) stay RESIDENT in shared memory for the life of the CTA;
//   * the input patch of a tile is loaded ONCE with its halo ([18 rows][16 pixel slots] x 64 ch, 36 KB) and the nine
//     taps are nine shifted UMMA-descriptor views of it (start = patch + (ky*16 + kx)*128 B, SBO = 2048 B; the 128-byte
//     swizzle is a pure function of the shared-memory address, so no descriptor base-offset is needed -- verified in
//     profiles/r01_halo_variant_test.txt): DRAM traffic is exactly algorithmic (73 / 98 MB per 640x400 image);
//   * persistent CTAs (one per SM) with a ring of halo slots and double-buffered TMEM accumulators: the producer
//     prefetches the next tiles while the tensor core works and the eight epilogue warps drain the previous tile.
// What bounds it now is the MMA's own operand traffic: an SS-mode M = 128 x N = 64 x K = 16 MMA reads 4 KB (A) + 2 KB (B) from
// shared memory at 128 B/clk = 48 cycles for 32 cycles of tensor work (profiles/r01_umma_issue_probe.txt: same floor with
// two issuing warps and with cta_group::2), i.e. <= 67 % of the tensor peak.  To sit AT that bound the issuing thread runs
// from precomputed descriptor words, running counters, probes of the next tile's barriers issued before the current MMAs,
// and a uniform-register accumulator address (9 instructions per MMA).
// Optional extras of the dgrad: the ReLU-mask activation tile of the layer below is TMA-loaded once per tile and used
// both as the A operand of the fused Gram-backward block (x D_b) and as the epilogue mask.
#include <algorithm>

#include "isx_common.cuh"
#include "isx_internal.h"
#include "isx_kernels.h"

namespace isx {

static constexpr int kC64Threads = 64 + 256;
static constexpr int kHalo = 18 * 16 * 128;   // bytes of one halo patch
static constexpr int kTile = 128 * 128;       // bytes of a 128-row x 64-channel bf16 tile

struct C64Params {
  int B, H, W, Cout;
  int tiles_x, tiles_y;
  long total_items;
  int halo_slots;
  int relu, fuse_pool, use_mask, use_gram;
  const float* bias;
  const __nv_bfloat16* add_buf;
  const float* aff_a;
  const float* aff_b;
  float* dx_nchw;
  int xc;
  const float* in_mask;
  int mask_b;
  uint8_t* pool_idx;
  int skip_out;
};

// smem carve-up (all offsets multiples of 1024)
struct C64Layout {
  int w, d, halo, act, stg, pstg, bars, total;
};
template <int BN, int EPI>
__host__ __device__ inline C64Layout c64_layout(int halo_slots, int use_mask, int use_gram, int fuse_pool) {
  C64Layout L;
  int off = 0;
  L.w = off; off += ((9 * BN * 128 + 1023) / 1024) * 1024;
  L.d = off; off += use_gram ? 2 * ((BN * 128 + 1023) / 1024) * 1024 : 0;
  L.halo = off; off += halo_slots * kHalo;
  L.act = off; off += use_mask ? 2 * kTile : 0;
  L.stg = off; off += EPI == 0 ? 2 * kTile : 0;
  L.pstg = off; off += fuse_pool ? 2 * 4096 : 0;
  L.bars = off; off += 512;
  L.total = off;
  return L;
}

// The tiles of a persistent CTA: w = first, first + stride, ... decomposed into (image b, tile r within the image)
// incrementally -- no 64-bit division per tile.
struct TileWalk {
  int b, r, stride, per_img, tiles_x;
  __device__ TileWalk(int first, int stride_, int per_img_, int tiles_x_)
      : b(first / per_img_), r(first % per_img_), stride(stride_), per_img(per_img_), tiles_x(tiles_x_) {}
  __device__ void next() {
    r += stride;
    while (r >= per_img) { r -= per_img; ++b; }
  }
  __device__ int x0() const { return (r % tiles_x) * 8; }
  __device__ int y0() const { return (r / tiles_x) * 16; }
};

template <int BN, int EPI>
__global__ void __launch_bounds__(kC64Threads, 1)
conv_c64_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmW,
                const __grid_constant__ CUtensorMap tmO, const __grid_constant__ CUtensorMap tmM,
                const __grid_constant__ CUtensorMap tmD, const __grid_constant__ CUtensorMap tmP, const C64Params p) {
  constexpr int kWSlab = BN * 128;
  constexpr int kAccCols = BN < 32 ? 32 : BN;
  constexpr int kTmemCols = 2 * kAccCols <= 32 ? 32 : 2 * kAccCols <= 64 ? 64 : 2 * kAccCols <= 128 ? 128 : 256;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const C64Layout L = c64_layout<BN, EPI>(p.halo_slots, p.use_mask, p.use_gram, p.fuse_pool);
  const int HS = p.halo_slots;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + L.bars);
  uint64_t* w_full = bars;                 // [1]
  uint64_t* halo_full = bars + 1;          // [4]
  uint64_t* halo_empty = bars + 5;         // [4]
  uint64_t* act_full = bars + 9;           // [2]
  uint64_t* act_empty = bars + 11;         // [2]
  uint64_t* d_full = bars + 13;            // [2]
  uint64_t* d_empty = bars + 15;           // [2]
  uint64_t* tmem_full = bars + 17;         // [2]
  uint64_t* tmem_empty = bars + 19;        // [2]
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(bars + 21);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmW);
    if (EPI == 0) tma_prefetch_desc(&tmO);
    if (p.use_mask) tma_prefetch_desc(&tmM);
    if (p.use_gram) tma_prefetch_desc(&tmD);
    if (p.fuse_pool) tma_prefetch_desc(&tmP);
    mbar_init(w_full, 1);
    for (int i = 0; i < 4; ++i) { mbar_init(&halo_full[i], 1); mbar_init(&halo_empty[i], 1); }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&act_full[i], 1);
      mbar_init(&act_empty[i], 8);   // one arrival per epilogue warp
      mbar_init(&d_full[i], 1);
      mbar_init(&d_empty[i], 1);
      mbar_init(&tmem_full[i], 1);
      mbar_init(&tmem_empty[i], 8);
    }
    fence_barrier_init();
  }
  // The persistent CTA owns its SM: it allocates ALL 512 TMEM columns, whatever it uses.  The allocation can then only succeed
  // once nobody else holds tensor memory on this SM, so the base is column 0 by construction (the MMA loop relies on
  // compile-time accumulator addresses) and a foreign tcgen05 kernel on another stream makes this CTA wait, not fault.
  if (warp == 1) tmem_alloc<512>(tmem_ptr_smem);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;
  const int total = static_cast<int>(p.total_items);  // < 2^31 (checked at launch)
  const int per_img = p.tiles_x * p.tiles_y;
  const int n_my = (total - static_cast<int>(blockIdx.x) + static_cast<int>(gridDim.x) - 1) / static_cast<int>(gridDim.x);

  if (warp == 0) {
    // ================================ TMA producer =========================================
    if (lane == 0) {
      mbar_arrive_expect_tx(w_full, 9 * kWSlab);
      for (int tap = 0; tap < 9; ++tap) tma_load_2d(smem + L.w + tap * kWSlab, &tmW, w_full, 0, tap * p.Cout);
      TileWalk tw(blockIdx.x, gridDim.x, per_img, p.tiles_x);
      uint32_t hs = 0, hph = 0, as = 0, aph = 0;
      for (int i = 0; i < n_my; ++i, tw.next()) {
        const int b = tw.b, x0 = tw.x0(), y0 = tw.y0();
        mbar_wait(&halo_empty[hs], hph ^ 1);
        mbar_arrive_expect_tx(&halo_full[hs], kHalo);
        tma_load_4d(smem + L.halo + hs * kHalo, &tmA, &halo_full[hs], 0, x0 - 1, y0 - 1, b);
        if (++hs == static_cast<uint32_t>(HS)) { hs = 0; hph ^= 1; }
        if (p.use_mask) {
          mbar_wait(&act_empty[as], aph ^ 1);
          mbar_arrive_expect_tx(&act_full[as], kTile);
          tma_load_4d(smem + L.act + as * kTile, &tmM, &act_full[as], 0, x0, y0, b);
        }
        if (p.use_gram) {
          mbar_wait(&d_empty[as], aph ^ 1);
          mbar_arrive_expect_tx(&d_full[as], kWSlab);
          tma_load_2d(smem + L.d + as * ((kWSlab + 1023) / 1024) * 1024, &tmD, &d_full[as], 0, b * p.Cout);
        }
        as ^= 1;
        if (as == 0) aph ^= 1;
      }
    }
  } else if (warp == 1) {
    // ================================ MMA issuer ===========================================
    if (lane == 0) {
      constexpr uint32_t idesc = umma_idesc_bf16(128, BN, false, false);
      // One CTA per SM owns the whole TMEM, so the allocation starts at column 0.  Using that constant (instead of the
      // value read back from shared memory) lets the accumulator address live in a uniform register: ptxas otherwise wraps
      // every tcgen05.mma in an ELECT / R2UR.BROADCAST / BRA.U.ANY waterfall (5 extra instructions per MMA on the
      // issue-bound thread).
      if (tmem_base != 0) {
        printf("isx: unexpected TMEM base %u (block %d)\n", tmem_base, blockIdx.x);
        __trap();
      }
      mbar_wait(w_full, 0);
      const uint64_t dw0 = umma_desc_sw128(smem_u32(smem + L.w), 16, 1024);
      const uint64_t da0 = umma_desc_sw128(smem_u32(smem + L.halo), 16, 2048);
      const uint32_t w_lo = static_cast<uint32_t>(dw0), w_hi = static_cast<uint32_t>(dw0 >> 32);
      const uint32_t a_lo0 = static_cast<uint32_t>(da0), a_hi = static_cast<uint32_t>(da0 >> 32);
      // Gram block operands: plain 128-row tiles (SBO 1024, same high word as the weight descriptor)
      constexpr int kDSlab = ((kWSlab + 1023) / 1024) * 1024;
      const uint32_t act_lo0 = static_cast<uint32_t>(umma_desc_sw128(smem_u32(smem + L.act), 16, 1024));
      const uint32_t d_lo0 = static_cast<uint32_t>(umma_desc_sw128(smem_u32(smem + L.d), 16, 1024));
      // running ring / phase counters: no division, no 64-bit arithmetic on the issuing thread's critical path
      uint32_t hs = 0, hph = 0, acc = 0, aph = 0, a_lo = a_lo0;
      bool t_ready = false, h_ready = false;  // probes of the NEXT tile's barriers, issued before this tile's MMAs
      for (int i = 0; i < n_my; ++i) {
        if (!t_ready) mbar_wait(&tmem_empty[acc], aph ^ 1);
        if (!h_ready) mbar_wait(&halo_full[hs], hph);
        tc_fence_after();
        const uint32_t d_tm = acc * kAccCols;  // TMEM base is 0 (checked above): keeps the address in a uniform register
        {
          const uint32_t hs_n = hs + 1 == static_cast<uint32_t>(HS) ? 0 : hs + 1;
          const uint32_t hph_n = hs_n == 0 ? hph ^ 1 : hph;
          t_ready = mbar_try_wait(&tmem_empty[acc ^ 1], acc == 1 ? aph : aph ^ 1);
          h_ready = mbar_try_wait(&halo_full[hs_n], hph_n);
        }
#pragma unroll
        for (int tap = 0; tap < 9; ++tap) {
          const int ky = tap / 3, kx = tap - ky * 3;
#pragma unroll
          for (int k = 0; k < 4; ++k)  // tap (ky, kx) = the halo patch shifted by ky rows and kx pixels
            umma_bf16_lohi(d_tm, a_lo + (((ky * 16 + kx) * 128 + k * 32) >> 4), a_hi, w_lo + ((tap * kWSlab + k * 32) >> 4), w_hi,
                           idesc, (tap | k) != 0 ? 1u : 0u);
        }
        umma_commit(&halo_empty[hs]);
        if (p.use_gram) {  // + act . D_b
          mbar_wait2(&act_full[acc], aph, &d_full[acc], aph);
          tc_fence_after();
          const uint32_t a2_lo = act_lo0 + acc * (kTile >> 4), b2_lo = d_lo0 + acc * (kDSlab >> 4);
#pragma unroll
          for (int k = 0; k < 4; ++k)
            umma_bf16_lohi(d_tm, a2_lo + 2 * k, w_hi, b2_lo + 2 * k, w_hi, idesc, 1u);
          umma_commit(&d_empty[acc]);
        }
        umma_commit(&tmem_full[acc]);
        a_lo += kHalo >> 4;
        if (++hs == static_cast<uint32_t>(HS)) { hs = 0; hph ^= 1; a_lo = a_lo0; }
        acc ^= 1;
        if (acc == 0) aph ^= 1;
      }
    }
  } else {
    // ================================ epilogue (8 warps) ===================================
    const int q = warp & 3;
    const int hsel = (warp - 2) >> 2;
    const int row = q * 32 + lane;
    const int tw = row & 7, th = row >> 3;
    TileWalk tiles(blockIdx.x, gridDim.x, per_img, p.tiles_x);
    uint32_t it = 0, gc = 0;
    for (int i = 0; i < n_my; ++i, ++it, tiles.next()) {
      const int b = tiles.b, x0 = tiles.x0(), y0 = tiles.y0();
      const uint32_t acc = it & 1;
      const int as = it & 1;
      const uint32_t d_tm = tmem_base + acc * kAccCols + (static_cast<uint32_t>(q * 32) << 16);
      const int x = x0 + tw, y = y0 + th;
      const bool valid = (x < p.W) && (y < p.H);
      mbar_wait(&tmem_full[acc], (it >> 1) & 1);
      tc_fence_after();
      if constexpr (EPI == 1) {
        if (hsel == 0) {
          uint32_t v[16];
          tmem_ld_32x16(d_tm, v);
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
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&tmem_empty[acc]);
      } else {
        const size_t pix = valid ? ((static_cast<size_t>(b) * p.H + y) * p.W + x) * p.Cout : 0;
        if (p.use_mask) mbar_wait(&act_full[as], (it >> 1) & 1);
        const uint8_t* mrow = smem + L.act + as * kTile + row * 128;
        const uint32_t slot = gc & 1;
        uint8_t* stg = smem + L.stg + slot * kTile;
        {
          const int h = hsel;
          const int n = h * 32;
          uint32_t v[32];
          tmem_ld_32x32(d_tm + n, v);
          tmem_ld_wait();
          // accumulator read: hand the TMEM set back to the MMA warp as early as possible
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(&tmem_empty[acc]);
          float f[32];
#pragma unroll
          for (int i = 0; i < 32; ++i) f[i] = __uint_as_float(v[i]);
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
          if (p.use_mask) {
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
            __syncwarp();
            if (lane == 0) mbar_arrive(&act_empty[as]);  // this warp is done with the activation tile
          }
          if (p.relu) {
#pragma unroll
            for (int i = 0; i < 32; ++i) f[i] = fmaxf(f[i], 0.f);
          }
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
        // staging slot (gc+1)&1 is written by the next tile: its TMA stores must have finished reading shared memory
        if (threadIdx.x == 64) tma_store_wait_read<0>();
        asm volatile("bar.sync 1, 256;" ::: "memory");
        if (threadIdx.x == 64 && !p.skip_out) {
          tma_store_4d(&tmO, stg, 0, x0, y0, b);
          tma_store_commit();
        }
        if (p.fuse_pool) {
          uint8_t* pst = smem + L.pstg + slot * 4096;
          const int item = threadIdx.x - 64;  // 0..255: 32 pooled pixels x 8 chunks
          const int pr = item >> 3, chunk = item & 7;
          const int px = pr & 3, py = pr >> 2;  // pooled tile is 4 x 8
          const int r00 = (2 * py) * 8 + 2 * px;
          const int rr[4] = {r00, r00 + 1, r00 + 8, r00 + 9};
          uint4 u4[4];
#pragma unroll
          for (int k = 0; k < 4; ++k) u4[k] = *reinterpret_cast<const uint4*>(stg + rr[k] * 128 + ((chunk ^ (rr[k] & 7)) * 16));
          uint4 m4;
          uint2 codes;
          pool4_codes(u4, m4, codes);
          if (p.pool_idx != nullptr) {  // routing bytes of the max-pool + ReLU backward, straight to global memory
            const int xp = (x0 >> 1) + px, yp = (y0 >> 1) + py;
            if (xp < (p.W >> 1) && yp < (p.H >> 1))
              *reinterpret_cast<uint2*>(p.pool_idx + ((static_cast<size_t>(b) * (p.H >> 1) + yp) * (p.W >> 1) + xp) * p.Cout +
                                        chunk * 8) = codes;
          }
          *reinterpret_cast<uint4*>(pst + pr * 128 + ((chunk ^ (pr & 7)) * 16)) = m4;
          fence_proxy_async_smem();
          asm volatile("bar.sync 1, 256;" ::: "memory");
          if (threadIdx.x == 64) {
            tma_store_4d(&tmP, pst, 0, x0 >> 1, y0 >> 1, b);
            tma_store_commit();
          }
        }
        ++gc;
      }
    }
    if (EPI == 0 && threadIdx.x == 64) tma_store_wait_all<0>();
    tc_fence_before();
  }
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc<512>(tmem_base);
  }
}


template <int BN, int EPI>
static int launch_c64(const ConvArgs& a, cudaStream_t stream) {
  C64Params p;
  memset(&p, 0, sizeof(p));
  p.B = a.B; p.H = a.H; p.W = a.W; p.Cout = a.Cout;
  p.tiles_x = (a.W + 7) / 8;
  p.tiles_y = (a.H + 15) / 16;
  p.total_items = static_cast<long>(p.tiles_x) * p.tiles_y * a.B;
  ISX_REQUIRE(p.total_items < (1L << 31) - kNumSMs, "conv_c64: too many tiles");
  p.relu = a.relu; p.bias = a.bias; p.add_buf = a.add_buf; p.aff_a = a.aff_a; p.aff_b = a.aff_b;
  p.use_mask = (EPI == 0 && a.mask_act != nullptr) ? 1 : 0;
  p.use_gram = (EPI == 0 && a.gram_act != nullptr) ? 1 : 0;
  ISX_REQUIRE(!p.use_gram || a.gram_act == a.mask_act, "conv_c64: the fused Gram operand must be the ReLU-mask activation");
  p.fuse_pool = (EPI == 0 && a.pool_out != nullptr && a.H >= 2 && a.W >= 2) ? 1 : 0;
  p.pool_idx = p.fuse_pool ? a.pool_idx : nullptr;
  p.skip_out = (p.fuse_pool && a.pool_idx != nullptr && a.skip_out) ? 1 : 0;
  p.dx_nchw = a.dx_nchw; p.xc = a.xc; p.in_mask = a.in_mask; p.mask_b = a.mask_b;
  int hs = 4;
  C64Layout L = c64_layout<BN, EPI>(hs, p.use_mask, p.use_gram, p.fuse_pool);
  const int cap = (227 - std::max(0, std::min(isx_ctx()->opt_smem_reserve_kb, 22))) * 1024;  // see conv_halo.cu
  while (hs > 2 && 1024 + L.total > cap) { --hs; L = c64_layout<BN, EPI>(hs, p.use_mask, p.use_gram, p.fuse_pool); }
  ISX_REQUIRE(1024 + L.total <= 227 * 1024, "conv_c64: %d B of shared memory exceed 227 KB", 1024 + L.total);
  p.halo_slots = hs;
  // At least 204 KB, so that no other TMEM-using CTA of this library (the conv1_1 head needs 29 KB, everything else more)
  // can share the SM when jobs run on several streams: the MMA thread relies on owning TMEM from column 0.
  const size_t smem_bytes = std::max<size_t>(1024 + L.total, 204 * 1024);

  CUtensorMap tmA, tmW, tmO, tmM, tmD, tmP;
  {
    uint64_t dims[4] = {64, (uint64_t)a.W, (uint64_t)a.H, (uint64_t)a.B};
    uint64_t str[3] = {128, (uint64_t)a.W * 128, (uint64_t)a.H * a.W * 128};
    uint32_t box[4] = {64, 16, 18, 1};
    if (isx_make_tmap_bf16(&tmA, a.in, 4, dims, str, box, true)) return 3;
  }
  {
    uint64_t dims[2] = {64, (uint64_t)9 * a.Cout};
    uint64_t str[1] = {128};
    uint32_t box[2] = {64, (uint32_t)BN};
    if (isx_make_tmap_bf16(&tmW, a.weight, 2, dims, str, box, true)) return 3;
  }
  tmO = tmA; tmM = tmA; tmD = tmW; tmP = tmA;
  if (EPI == 0) {
    uint64_t dims[4] = {(uint64_t)a.Cout, (uint64_t)a.W, (uint64_t)a.H, (uint64_t)a.B};
    uint64_t str[3] = {(uint64_t)a.Cout * 2, (uint64_t)a.W * a.Cout * 2, (uint64_t)a.H * a.W * a.Cout * 2};
    uint32_t box[4] = {64, 8, 16, 1};
    if (isx_make_tmap_bf16(&tmO, a.out, 4, dims, str, box, true)) return 3;
    if (p.use_mask && isx_make_tmap_bf16(&tmM, a.mask_act, 4, dims, str, box, true)) return 3;
    if (p.use_gram) {
      uint64_t d2[2] = {(uint64_t)a.Cout, (uint64_t)a.Cout * a.B};
      uint64_t s2[1] = {(uint64_t)a.Cout * 2};
      uint32_t b2[2] = {64, (uint32_t)BN};
      if (isx_make_tmap_bf16(&tmD, a.gram_D, 2, d2, s2, b2, true)) return 3;
    }
    if (p.fuse_pool) {
      uint64_t dp[4] = {(uint64_t)a.Cout, (uint64_t)(a.W / 2), (uint64_t)(a.H / 2), (uint64_t)a.B};
      uint64_t sp[3] = {(uint64_t)a.Cout * 2, (uint64_t)(a.W / 2) * a.Cout * 2, (uint64_t)(a.H / 2) * (a.W / 2) * a.Cout * 2};
      uint32_t bp[4] = {64, 4, 8, 1};
      if (isx_make_tmap_bf16(&tmP, a.pool_out, 4, dp, sp, bp, true)) return 3;
    }
  }
  auto kern = conv_c64_kernel<BN, EPI>;
  ISX_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bytes));
  const long grid = std::min<long>(p.total_items, kNumSMs);
  isx_prof_begin(ISX_PROF_CONV, 2.0 * (9 * 64 + (p.use_gram ? a.Cout : 0)) * a.Cout * static_cast<double>(a.B) * a.H * a.W, stream);
  kern<<<(unsigned)grid, kC64Threads, smem_bytes, stream>>>(tmA, tmW, tmO, tmM, tmD, tmP, p);
  isx_prof_end(ISX_PROF_CONV, stream);
  ISX_LAUNCH_CHECK();
  return 0;
}

// Cin = 64, 3x3, shared weights, Cout 64 (bf16 NHWC out) or the N = 16 image-gradient tail.
bool conv_c64_applicable(const ConvArgs& a) {
  if (a.Cin != 64 || a.ntaps != 9 || a.per_image_weights || a.stride != 1) return false;
  if (a.dx_nchw != nullptr) return a.Cout == 16;
  if (a.Cout != 64) return false;
  if (a.gram_act != nullptr && a.gram_act != a.mask_act) return false;
  return true;
}

int conv_c64(const ConvArgs& a, cudaStream_t stream) {
  ISX_REQUIRE(conv_c64_applicable(a), "conv_c64: not applicable");
  if (a.dx_nchw != nullptr) return launch_c64<16, 1>(a, stream);
  return launch_c64<64, 0>(a, stream);
}

}  // namespace isx
