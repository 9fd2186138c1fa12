// 3x3 convolutions of the mid layers (conv2_x, conv3_x: Cin >= 64, Cout a multiple of 64/128) with HALF the L2 -> shared
// memory operand traffic of the generic kernel.  Measured on the generic kernel (profiles/r01_operand_skip_probe.txt):
// skipping its TMA operand loads lifts conv2_2 from 1110 to 1414 TFLOP/s and conv3_2 from 1354 to 1685 -- it is bound
// by operand delivery (~96 B/clk/SM: every tap re-loads its 2 x 16 KB A tiles), not by the tensor pipe.  This variant:
//   * one work item = a PAIR of 128-pixel tiles (16x16 or 8x32 pixels) x 128 (or 64) output channels;
//   * per 64-channel input block the pair's patch is loaded ONCE with its halo (18x18 or 10x34 pixel rows of 128 B) and
//     the nine taps of both tiles are shifted UMMA-descriptor views of it (SBO = patch pitch; the 128-byte swizzle is a
//     function of the shared-memory address only, see conv_c64.cu) -- A traffic drops from 9 x 32 KB to ~42 KB;
//   * the weight slab of a tap (BN x 64) streams through its own ring and feeds BOTH tiles (8 MMAs per slab);
//   * persistent CTAs (one per SM), two TMEM accumulator sets (2 x 2 x BN columns): the eight epilogue warps drain
//     item i while the tensor core runs item i+1; the MMA thread issues from precomputed descriptor words
//     (umma_bf16_lohi) with running ring counters;
//   * the epilogue walks the item as 128-row x 64-channel sub-tiles (bias / ReLU / residual add / ReLU mask /
//     BN-statistics affine term / fused 2x2 max-pool, staged in swizzled shared memory and written with TMA); the
//     ReLU-mask activation sub-tiles are TMA-loaded by the epilogue itself two sub-tiles ahead;
//   * the fused Gram backward (dX += act . D_b) runs as extra K blocks whose A operand is the plain activation tile.
#include <algorithm>

#include "isx_common.cuh"
#include "isx_internal.h"
#include "isx_kernels.h"

namespace isx {

static constexpr int kHaloThreads = 64 + 256;
static constexpr int kHaloSlot = 43 * 1024;  // >= 18*18*128 (41472) and 10*34*128 (43520); also holds two plain 16 KB tiles
static constexpr int kSub = 128 * 128;       // bytes of a 128-row x 64-channel bf16 sub-tile

struct HaloParams {
  int B, H, W, Cin, Cout;
  int pairs_x, pairs_y, n_tiles;
  int total_items;
  int cin_blocks, extra_kb;
  int w_stages;
  int relu, fuse_pool, use_mask;
  const float* bias;
  const __nv_bfloat16* add_buf;
  const float* aff_a;
  const float* aff_b;
  uint8_t* pool_idx;
  int skip_out;
};

struct HaloLayout {
  int halo, w, act, stg, pstg, bars, total;
};
template <int BN>
__host__ __device__ inline HaloLayout halo_layout(int w_stages, int use_mask, int fuse_pool) {
  HaloLayout L;
  int off = 0;
  L.halo = off; off += 2 * kHaloSlot;
  L.w = off; off += w_stages * BN * 128;
  L.act = off; off += use_mask ? 2 * kSub : 0;
  L.stg = off; off += 2 * kSub;
  L.pstg = off; off += fuse_pool ? 2 * 4096 : 0;
  L.bars = off; off += 512;
  L.total = off;
  return L;
}

// Work items of a persistent CTA: w = first, first + stride, ...; w -> (image, pair row, pair column, Cout tile) with
// the Cout tile fastest, so the CTAs running at the same time share the pair's input patch in L2.
template <bool VERT>
struct ItemWalk {
  int b, r, stride, per_img, pairs_x, n_tiles;
  __device__ ItemWalk(int first, int stride_, int per_img_, int pairs_x_, int n_tiles_)
      : b(first / per_img_), r(first % per_img_), stride(stride_), per_img(per_img_), pairs_x(pairs_x_), n_tiles(n_tiles_) {}
  __device__ void next() {
    r += stride;
    while (r >= per_img) { r -= per_img; ++b; }
  }
  __device__ int nt() const { return r % n_tiles; }
  __device__ int x0() const { return ((r / n_tiles) % pairs_x) * (VERT ? 8 : 16); }
  __device__ int y0() const { return ((r / n_tiles) / pairs_x) * (VERT ? 32 : 16); }
};

template <int BN, bool VERT>
__global__ void __launch_bounds__(kHaloThreads, 1)
conv_halo_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmW,
                 const __grid_constant__ CUtensorMap tmO, const __grid_constant__ CUtensorMap tmM,
                 const __grid_constant__ CUtensorMap tmA2, const __grid_constant__ CUtensorMap tmD,
                 const __grid_constant__ CUtensorMap tmP, const HaloParams p) {
  constexpr int kPitch = VERT ? 10 : 18;                 // pixels per patch row
  constexpr int kPatchRows = VERT ? 34 : 18;
  constexpr int kHaloBytes = kPitch * kPatchRows * 128;
  constexpr int kMtOff = VERT ? 16 * kPitch * 128 : 8 * 128;  // second tile of the pair inside the patch
  constexpr int kWStage = BN * 128;
  constexpr int kNH = BN / 64;                            // 64-channel sub-tiles per 128-pixel tile
  constexpr int kNSub = 2 * kNH;
  constexpr int kAccCols = 2 * BN;                        // one accumulator set: two tiles x BN columns
  constexpr int kTmemCols = 2 * kAccCols;                 // 256 (BN = 64) or 512 (BN = 128)
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const HaloLayout L = halo_layout<BN>(p.w_stages, p.use_mask, p.fuse_pool);
  const int WS = p.w_stages;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + L.bars);
  uint64_t* halo_full = bars;          // [2]
  uint64_t* halo_empty = bars + 2;     // [2]
  uint64_t* w_full = bars + 4;         // [8]
  uint64_t* w_empty = bars + 12;       // [8]
  uint64_t* act_full = bars + 20;      // [2]
  uint64_t* tmem_full = bars + 22;     // [2]
  uint64_t* tmem_empty = bars + 24;    // [2]
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(bars + 26);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmW);
    tma_prefetch_desc(&tmO);
    if (p.use_mask) tma_prefetch_desc(&tmM);
    if (p.extra_kb > 0) { tma_prefetch_desc(&tmA2); tma_prefetch_desc(&tmD); }
    if (p.fuse_pool) tma_prefetch_desc(&tmP);
    for (int i = 0; i < 2; ++i) {
      mbar_init(&halo_full[i], 1);
      mbar_init(&halo_empty[i], 1);
      mbar_init(&act_full[i], 1);
      mbar_init(&tmem_full[i], 1);
      mbar_init(&tmem_empty[i], 8);  // one arrival per epilogue warp
    }
    for (int i = 0; i < 8; ++i) { mbar_init(&w_full[i], 1); mbar_init(&w_empty[i], 1); }
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
  const int per_img = p.pairs_x * p.pairs_y * p.n_tiles;
  const int n_my = (p.total_items - static_cast<int>(blockIdx.x) + static_cast<int>(gridDim.x) - 1) / static_cast<int>(gridDim.x);

  if (warp == 0) {
    // ================================ TMA producer =========================================
    if (lane == 0) {
      ItemWalk<VERT> it(blockIdx.x, gridDim.x, per_img, p.pairs_x, p.n_tiles);
      uint32_t hs = 0, hph = 0, ws = 0, wph = 0;
      for (int i = 0; i < n_my; ++i, it.next()) {
        const int b = it.b, x0 = it.x0(), y0 = it.y0(), n0 = it.nt() * BN;
        for (int c = 0; c < p.cin_blocks; ++c) {
          mbar_wait(&halo_empty[hs], hph ^ 1);
          mbar_arrive_expect_tx(&halo_full[hs], kHaloBytes);
          tma_load_4d(smem + L.halo + hs * kHaloSlot, &tmA, &halo_full[hs], c * 64, x0 - 1, y0 - 1, b);
          hs ^= 1;
          if (hs == 0) hph ^= 1;
          for (int tap = 0; tap < 9; ++tap) {
            mbar_wait(&w_empty[ws], wph ^ 1);
            mbar_arrive_expect_tx(&w_full[ws], kWStage);
            tma_load_2d(smem + L.w + ws * kWStage, &tmW, &w_full[ws], c * 64, tap * p.Cout + n0);
            if (++ws == static_cast<uint32_t>(WS)) { ws = 0; wph ^= 1; }
          }
        }
        for (int c2 = 0; c2 < p.extra_kb; ++c2) {  // fused Gram backward: A = the two plain activation tiles, B = D_b
          mbar_wait(&halo_empty[hs], hph ^ 1);
          mbar_arrive_expect_tx(&halo_full[hs], 2 * kSub);
          uint8_t* slot = smem + L.halo + hs * kHaloSlot;
          tma_load_4d(slot, &tmA2, &halo_full[hs], c2 * 64, x0, y0, b);
          tma_load_4d(slot + kSub, &tmA2, &halo_full[hs], c2 * 64, VERT ? x0 : x0 + 8, VERT ? y0 + 16 : y0, b);
          hs ^= 1;
          if (hs == 0) hph ^= 1;
          mbar_wait(&w_empty[ws], wph ^ 1);
          mbar_arrive_expect_tx(&w_full[ws], kWStage);
          tma_load_2d(smem + L.w + ws * kWStage, &tmD, &w_full[ws], c2 * 64, b * p.Cout + n0);
          if (++ws == static_cast<uint32_t>(WS)) { ws = 0; wph ^= 1; }
        }
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
      const uint64_t dh = umma_desc_sw128(smem_u32(smem + L.halo), 16, kPitch * 128);  // shifted views of the patch
      const uint64_t dp = umma_desc_sw128(smem_u32(smem + L.halo), 16, 1024);          // plain 128-row tiles / weight slabs
      const uint64_t dw = umma_desc_sw128(smem_u32(smem + L.w), 16, 1024);
      const uint32_t h_lo0 = static_cast<uint32_t>(dh), h_hi = static_cast<uint32_t>(dh >> 32);
      const uint32_t p_hi = static_cast<uint32_t>(dp >> 32);
      const uint32_t w_lo0 = static_cast<uint32_t>(dw), w_hi = static_cast<uint32_t>(dw >> 32);
      uint32_t hs = 0, hph = 0, ws = 0, wph = 0, acc = 0, aph = 0, b_lo = w_lo0;
      // An mbarrier probe costs ~150 cycles even when the phase completed long ago -- as much as two or three MMA issues.
      // The probe of the NEXT weight stage is therefore issued before the current tap's MMAs and consumed after them.
      bool w_ready = false, h_ready = false;
      auto next_stage = [&]() {
        b_lo += kWStage >> 4;
        if (++ws == static_cast<uint32_t>(WS)) { ws = 0; wph ^= 1; b_lo = w_lo0; }
      };
      for (int i = 0; i < n_my; ++i) {
        mbar_wait(&tmem_empty[acc], aph ^ 1);
        tc_fence_after();
        const uint32_t d_tm = acc * kAccCols;  // TMEM base is 0 (checked above): keeps the address in a uniform register
        for (int c = 0; c < p.cin_blocks; ++c) {
          if (!h_ready) mbar_wait(&halo_full[hs], hph);
          h_ready = false;
          const uint32_t a_lo = h_lo0 + hs * (kHaloSlot >> 4);
#pragma unroll
          for (int tap = 0; tap < 9; ++tap) {
            const int ky = tap / 3, kx = tap - ky * 3;
            if (!w_ready) mbar_wait(&w_full[ws], wph);
            tc_fence_after();
            const uint32_t b_cur = b_lo;
            const uint32_t ws_cur = ws;
            next_stage();
            w_ready = mbar_try_wait(&w_full[ws], wph);
            if (tap == 8) h_ready = mbar_try_wait(&halo_full[hs ^ 1], hs == 1 ? hph ^ 1 : hph);  // next patch slot
#pragma unroll
            for (int mt = 0; mt < 2; ++mt) {
#pragma unroll
              for (int k = 0; k < 4; ++k)
                umma_bf16_lohi(d_tm + mt * BN, a_lo + (((ky * kPitch + kx) * 128 + mt * kMtOff + k * 32) >> 4), h_hi,
                               b_cur + 2 * k, w_hi, idesc, (tap | k) != 0 ? 1u : (c != 0 ? 1u : 0u));
            }
            umma_commit(&w_empty[ws_cur]);
          }
          umma_commit(&halo_empty[hs]);
          hs ^= 1;
          if (hs == 0) hph ^= 1;
        }
        for (int c2 = 0; c2 < p.extra_kb; ++c2) {
          if (!h_ready) mbar_wait(&halo_full[hs], hph);
          h_ready = false;
          if (!w_ready) mbar_wait(&w_full[ws], wph);
          tc_fence_after();
          const uint32_t a_lo = h_lo0 + hs * (kHaloSlot >> 4);
          const uint32_t b_cur = b_lo;
          const uint32_t ws_cur = ws;
          next_stage();
          w_ready = mbar_try_wait(&w_full[ws], wph);
#pragma unroll
          for (int mt = 0; mt < 2; ++mt) {
#pragma unroll
            for (int k = 0; k < 4; ++k)
              umma_bf16_lohi(d_tm + mt * BN, a_lo + ((mt * kSub + k * 32) >> 4), p_hi, b_cur + 2 * k, w_hi, idesc, 1u);
          }
          umma_commit(&w_empty[ws_cur]);
          umma_commit(&halo_empty[hs]);
          hs ^= 1;
          if (hs == 0) hph ^= 1;
        }
        umma_commit(&tmem_full[acc]);
        acc ^= 1;
        if (acc == 0) aph ^= 1;
      }
    }
  } else {
    // ================================ epilogue (8 warps) ===================================
    const int q = warp & 3;             // TMEM lane quadrant of this warp
    const int hsel = (warp - 2) >> 2;   // which 32-column half of a 64-channel sub-tile
    const int row = q * 32 + lane;
    const int tw = row & 7, th = row >> 3;
    const bool leader = threadIdx.x == 64;
    ItemWalk<VERT> it(blockIdx.x, gridDim.x, per_img, p.pairs_x, p.n_tiles);
    // sub-tile s of an item: tile mt = s / kNH at (x0 + (VERT ? 0 : 8 mt), y0 + (VERT ? 16 mt : 0)), channels n0 + 64 (s % kNH)
    auto issue_mask_load = [&](const ItemWalk<VERT>& w, int s, uint32_t g) {
      const int mt = s / kNH, nh = s - mt * kNH;
      const uint32_t slot = g & 1;
      mbar_arrive_expect_tx(&act_full[slot], kSub);
      tma_load_4d(smem + L.act + slot * kSub, &tmM, &act_full[slot], w.nt() * BN + nh * 64,
                  w.x0() + (VERT ? 0 : 8 * mt), w.y0() + (VERT ? 16 * mt : 0), w.b);
    };
    uint32_t g = 0;  // running sub-tile counter: staging / activation slot = g & 1
    if (p.use_mask && leader && n_my > 0) {
      issue_mask_load(it, 0, 0);
      issue_mask_load(it, 1, 1);
    }
    uint32_t acc = 0, aph = 0;
    for (int i = 0; i < n_my; ++i) {
      const int b = it.b, x0 = it.x0(), y0 = it.y0(), n0 = it.nt() * BN;
      ItemWalk<VERT> nxt = it;
      nxt.next();
      mbar_wait(&tmem_full[acc], aph);
      tc_fence_after();
#pragma unroll 1
      for (int s = 0; s < kNSub; ++s, ++g) {
        const int mt = s / kNH, nh = s - mt * kNH;
        const int xs = x0 + (VERT ? 0 : 8 * mt), ys = y0 + (VERT ? 16 * mt : 0);
        const int nc = n0 + nh * 64 + hsel * 32;  // first of this thread's 32 output channels
        const int x = xs + tw, y = ys + th;
        const bool valid = (x < p.W) && (y < p.H);
        const size_t pix = valid ? ((static_cast<size_t>(b) * p.H + y) * p.W + x) * p.Cout : 0;
        const uint32_t slot = g & 1;
        uint8_t* stg = smem + L.stg + slot * kSub;
        uint32_t v[32];
        tmem_ld_32x32(tmem_base + acc * kAccCols + mt * BN + nh * 64 + hsel * 32 + (static_cast<uint32_t>(q * 32) << 16), v);
        tmem_ld_wait();
        if (s == kNSub - 1) {  // accumulator set fully read: hand it back to the MMA warp
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(&tmem_empty[acc]);
        }
        float f[32];
#pragma unroll
        for (int j = 0; j < 32; ++j) f[j] = __uint_as_float(v[j]);
        if (p.bias != nullptr) {
#pragma unroll
          for (int j = 0; j < 32; j += 4) {
            const float4 bv = __ldg(reinterpret_cast<const float4*>(p.bias + nc + j));
            f[j] += bv.x; f[j + 1] += bv.y; f[j + 2] += bv.z; f[j + 3] += bv.w;
          }
        }
        if (p.add_buf != nullptr && valid) {
#pragma unroll
          for (int j = 0; j < 32; j += 8) {
            const uint4 u = __ldg(reinterpret_cast<const uint4*>(p.add_buf + pix + nc + j));
            float2 t;
            t = unpack_bf16x2(u.x); f[j] += t.x; f[j + 1] += t.y;
            t = unpack_bf16x2(u.y); f[j + 2] += t.x; f[j + 3] += t.y;
            t = unpack_bf16x2(u.z); f[j + 4] += t.x; f[j + 5] += t.y;
            t = unpack_bf16x2(u.w); f[j + 6] += t.x; f[j + 7] += t.y;
          }
        }
        if (p.use_mask) {
          mbar_wait(&act_full[slot], (g >> 1) & 1);
          const uint8_t* mrow = smem + L.act + slot * kSub + row * 128;
#pragma unroll
          for (int j = 0; j < 32; j += 8) {
            const int chunk = (hsel * 4 + (j >> 3)) ^ (row & 7);
            const uint4 u = *reinterpret_cast<const uint4*>(mrow + chunk * 16);
            float a[8];
            float2 t;
            t = unpack_bf16x2(u.x); a[0] = t.x; a[1] = t.y;
            t = unpack_bf16x2(u.y); a[2] = t.x; a[3] = t.y;
            t = unpack_bf16x2(u.z); a[4] = t.x; a[5] = t.y;
            t = unpack_bf16x2(u.w); a[6] = t.x; a[7] = t.y;
            if (p.aff_a != nullptr && valid) {
              const float* pa = p.aff_a + static_cast<size_t>(b) * p.Cout + nc + j;
              const float* pb = p.aff_b + static_cast<size_t>(b) * p.Cout + nc + j;
#pragma unroll
              for (int e = 0; e < 8; ++e) f[j + e] += __ldg(pa + e) + __ldg(pb + e) * a[e];
            }
#pragma unroll
            for (int e = 0; e < 8; ++e) f[j + e] = a[e] > 0.f ? f[j + e] : 0.f;
          }
        }
        if (p.relu) {
#pragma unroll
          for (int j = 0; j < 32; ++j) f[j] = fmaxf(f[j], 0.f);
        }
        uint8_t* rowp = stg + row * 128;
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          uint4 o;
          o.x = pack_bf16x2(f[c * 8 + 0], f[c * 8 + 1]);
          o.y = pack_bf16x2(f[c * 8 + 2], f[c * 8 + 3]);
          o.z = pack_bf16x2(f[c * 8 + 4], f[c * 8 + 5]);
          o.w = pack_bf16x2(f[c * 8 + 6], f[c * 8 + 7]);
          const int chunk = (hsel * 4 + c) ^ (row & 7);
          *reinterpret_cast<uint4*>(rowp + chunk * 16) = o;
        }
        fence_proxy_async_smem();
        // the other staging slot is rewritten by the next sub-tile: its TMA stores must have finished reading it
        if (leader) tma_store_wait_read<0>();
        asm volatile("bar.sync 1, 256;" ::: "memory");
        const bool inside = xs < p.W && ys < p.H;  // a tile of the pair may lie entirely outside the image
        if (leader) {
          if (inside && !p.skip_out) {
            tma_store_4d(&tmO, stg, n0 + nh * 64, xs, ys, b);
            tma_store_commit();
          }
          // every epilogue thread is past its reads of activation slot g & 1: refill it for sub-tile g + 2
          if (p.use_mask) {
            if (s + 2 < kNSub) issue_mask_load(it, s + 2, g + 2);
            else if (i + 1 < n_my) issue_mask_load(nxt, s + 2 - kNSub, g + 2);
          }
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
            const int xp = (xs >> 1) + px, yp = (ys >> 1) + py;
            if (xp < (p.W >> 1) && yp < (p.H >> 1))
              *reinterpret_cast<uint2*>(p.pool_idx + ((static_cast<size_t>(b) * (p.H >> 1) + yp) * (p.W >> 1) + xp) * p.Cout +
                                        n0 + nh * 64 + chunk * 8) = codes;
          }
          *reinterpret_cast<uint4*>(pst + pr * 128 + ((chunk ^ (pr & 7)) * 16)) = m4;
          fence_proxy_async_smem();
          asm volatile("bar.sync 1, 256;" ::: "memory");
          if (leader && inside) {
            tma_store_4d(&tmP, pst, n0 + nh * 64, xs >> 1, ys >> 1, b);
            tma_store_commit();
          }
        }
      }
      it = nxt;
      acc ^= 1;
      if (acc == 0) aph ^= 1;
    }
    if (leader) tma_store_wait_all<0>();
    tc_fence_before();
  }
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc<512>(tmem_base);
  }
}


template <int BN, bool VERT>
static int launch_halo(const ConvArgs& a, cudaStream_t stream) {
  HaloParams p;
  memset(&p, 0, sizeof(p));
  p.B = a.B; p.H = a.H; p.W = a.W; p.Cin = a.Cin; p.Cout = a.Cout;
  p.pairs_x = VERT ? (a.W + 7) / 8 : (a.W + 15) / 16;
  p.pairs_y = VERT ? (a.H + 31) / 32 : (a.H + 15) / 16;
  p.n_tiles = a.Cout / BN;
  const long total = static_cast<long>(p.pairs_x) * p.pairs_y * p.n_tiles * a.B;
  ISX_REQUIRE(total < (1L << 31) - kNumSMs, "conv_halo: too many work items");
  p.total_items = static_cast<int>(total);
  p.cin_blocks = a.Cin / 64;
  p.extra_kb = a.gram_act != nullptr ? a.Cout / 64 : 0;
  p.relu = a.relu; p.bias = a.bias; p.add_buf = a.add_buf; p.aff_a = a.aff_a; p.aff_b = a.aff_b;
  p.use_mask = a.mask_act != nullptr ? 1 : 0;
  p.fuse_pool = (a.pool_out != nullptr && a.H >= 2 && a.W >= 2) ? 1 : 0;
  p.pool_idx = p.fuse_pool ? a.pool_idx : nullptr;
  p.skip_out = (p.fuse_pool && a.pool_idx != nullptr && a.skip_out) ? 1 : 0;
  int ws = 6;
  HaloLayout L = halo_layout<BN>(ws, p.use_mask, p.fuse_pool);
  // "smem_reserve_kb" (<= 22): leave that much of the SM's shared memory free, so that one TMEM-free streaming CTA (the
  // L-BFGS passes of another stream) can be resident beside this persistent CTA and use the HBM bandwidth it leaves idle
  const int cap = (227 - std::max(0, std::min(isx_ctx()->opt_smem_reserve_kb, 22))) * 1024;
  while (ws > 2 && 1024 + L.total > cap) { --ws; L = halo_layout<BN>(ws, p.use_mask, p.fuse_pool); }
  ISX_REQUIRE(1024 + L.total <= 227 * 1024, "conv_halo: %d B of shared memory exceed 227 KB", 1024 + L.total);
  p.w_stages = ws;
  // At least 204 KB, so that no other TMEM-using CTA of this library (the conv1_1 head needs 29 KB, everything else more)
  // can share the SM when jobs run on several streams: the MMA thread relies on owning TMEM from column 0.
  const size_t smem_bytes = std::max<size_t>(1024 + L.total, 204 * 1024);

  CUtensorMap tmA, tmW, tmO, tmM, tmA2, tmD, tmP;
  {
    uint64_t dims[4] = {(uint64_t)a.Cin, (uint64_t)a.W, (uint64_t)a.H, (uint64_t)a.B};
    uint64_t str[3] = {(uint64_t)a.Cin * 2, (uint64_t)a.W * a.Cin * 2, (uint64_t)a.H * a.W * a.Cin * 2};
    uint32_t box[4] = {64, VERT ? 10u : 18u, VERT ? 34u : 18u, 1};
    if (isx_make_tmap_bf16(&tmA, a.in, 4, dims, str, box, true)) return 3;
  }
  {
    uint64_t dims[2] = {(uint64_t)a.Cin, (uint64_t)9 * a.Cout};
    uint64_t str[1] = {(uint64_t)a.Cin * 2};
    uint32_t box[2] = {64, (uint32_t)BN};
    if (isx_make_tmap_bf16(&tmW, a.weight, 2, dims, str, box, true)) return 3;
  }
  {
    uint64_t dims[4] = {(uint64_t)a.Cout, (uint64_t)a.W, (uint64_t)a.H, (uint64_t)a.B};
    uint64_t str[3] = {(uint64_t)a.Cout * 2, (uint64_t)a.W * a.Cout * 2, (uint64_t)a.H * a.W * a.Cout * 2};
    uint32_t box[4] = {64, 8, 16, 1};
    if (isx_make_tmap_bf16(&tmO, a.out, 4, dims, str, box, true)) return 3;
    tmM = tmO; tmA2 = tmO;
    if (p.use_mask && isx_make_tmap_bf16(&tmM, a.mask_act, 4, dims, str, box, true)) return 3;
    if (p.extra_kb > 0 && isx_make_tmap_bf16(&tmA2, a.gram_act, 4, dims, str, box, true)) return 3;
  }
  tmD = tmW; tmP = tmO;
  if (p.extra_kb > 0) {
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
  auto kern = conv_halo_kernel<BN, VERT>;
  ISX_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bytes));
  const int grid = std::min<int>(p.total_items, kNumSMs);
  isx_prof_begin(ISX_PROF_CONV, 2.0 * (9.0 * a.Cin + (p.extra_kb ? a.Cout : 0)) * a.Cout * static_cast<double>(a.B) * a.H * a.W, stream);
  kern<<<(unsigned)grid, kHaloThreads, smem_bytes, stream>>>(tmA, tmW, tmO, tmM, tmA2, tmD, tmP, p);
  isx_prof_end(ISX_PROF_CONV, stream);
  ISX_LAUNCH_CHECK();
  return 0;
}

// fraction of the computed pixels that lie inside the image for a pair shape
static double pair_efficiency(int H, int W, int pw, int ph) {
  const double cw = static_cast<double>((W + pw - 1) / pw) * pw, ch = static_cast<double>((H + ph - 1) / ph) * ph;
  return (static_cast<double>(W) / cw) * (static_cast<double>(H) / ch);
}

bool conv_halo_applicable(const ConvArgs& a) {
  if (a.ntaps != 9 || a.per_image_weights || a.dx_nchw != nullptr || a.stride != 1) return false;
  if (a.Cin % 64 != 0 || a.Cout % 64 != 0) return false;
  if (a.out == nullptr) return false;
  return true;
}

// 0: not worth it (few work items or mostly padding); otherwise 1 (16x16 pairs) or 2 (8x32 pairs)
int conv_halo_pick(const ConvArgs& a) {
  const double eh = pair_efficiency(a.H, a.W, 16, 16), ev = pair_efficiency(a.H, a.W, 8, 32);
  return ev > eh ? 2 : 1;
}
double conv_halo_efficiency(const ConvArgs& a) {
  return std::max(pair_efficiency(a.H, a.W, 16, 16), pair_efficiency(a.H, a.W, 8, 32));
}

int conv_halo(const ConvArgs& a, cudaStream_t stream) {
  ISX_REQUIRE(conv_halo_applicable(a), "conv_halo: not applicable");
  const bool vert = conv_halo_pick(a) == 2;
  if (a.Cout % 128 == 0) return vert ? launch_halo<128, true>(a, stream) : launch_halo<128, false>(a, stream);
  return vert ? launch_halo<64, true>(a, stream) : launch_halo<64, false>(a, stream);
}

}  // namespace isx
