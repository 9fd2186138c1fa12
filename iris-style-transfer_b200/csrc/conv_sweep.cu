// 3x3 convolutions with Cin = Cout = 64 (conv1_2 forward and dgrad) as a SWEEP with the taps of the sweep axis stacked in N.
//
// conv_c64.cu issues, per 128-pixel tile, 36 MMAs of M = 128 x N = 64 x K = 16 -- and an SS-mode MMA of that shape reads
// 4 KB (A) + 2 KB (B) from shared memory at 128 B/clk: 48 cycles for 32 cycles of tensor work, <= 67 % of the tensor peak
// whatever the issue loop does (profiles/r01_umma_issue_probe.txt).  The way out is a larger N, and N is not limited by the
// 64 output channels: one A view feeds several OUTPUT TILES at once when those tiles are shifted copies of each other.
//
//   * A tile is a STRIP: 128 consecutive pixels along one image axis (the strip axis u) at ONE coordinate v of the other
//     axis (the sweep axis).  The strip at sweep coordinate v, shifted by ku - 1 pixels along u, is the A operand of the taps
//     (ku, ks) of the three output strips v - 1, v, v + 1 (ks = 2, 1, 0): ONE MMA of N = 192 against the weight slab
//     [W(ku, ks=2) | W(ku, ks=1) | W(ku, ks=0)] accumulates into three neighbouring accumulators.  Per 128 pixels: 12 MMAs
//     of N = 192 (A 4 KB + B 6 KB = 80 clk of operand traffic for 96 clk of tensor work: tensor-bound) instead of 36 of N = 64.
//   * The accumulators live in a RING of eight 64-column slots that fills the whole TMEM (8 x 64 = 512 columns): output strip
//     number g of a CTA uses slot g & 7; an input strip touches three consecutive slots (the MMA is split in two where the
//     window wraps around the ring); the strip that receives its third contribution is committed to the epilogue, which
//     drains it while the sweep goes on -- no accumulator hand-over stall, ever.
//   * A CTA sweeps a segment of ~100 sweep coordinates of one (image, 128-pixel strip position): persistent CTAs, one per SM,
//     the strip patches ([130 pixels] x 64 ch with a one-pixel halo at both ends, the three ku taps are views shifted by one
//     128-byte row) come through a TMA ring, the nine weight slabs (72 KB) stay resident in shared memory.
//   * Either image axis can be the strip axis (the tensor maps present the NHWC tensor as (c, u, v, b)); the launcher picks
//     the one that wastes fewer of the 128 strip positions (640 = 5 x 128 rows for the 640 x 400 eye frames).
//   * Epilogue as in conv_c64 / conv_halo: bias / ReLU / residual add / ReLU mask / BN-affine term, bf16 tile staged in swizzled
//     shared memory and stored by TMA; fused 2x2 max-pool (two consecutive strips) with the routing bytes of its backward;
//     the dgrad's ReLU-mask activation strip doubles as the A operand of the fused Gram backward (x D_b, N = 64).
//
// STATUS (round 2, profiles/r02_conv_sweep_experiment.txt, profiles/r02_ab_sweep64.txt): the FORWARD launches run here by default
// (option "sweep64" = 1): 14.0-14.8 us per 640x400 image against 17.5-18.1 for conv_c64 (1 340 TFLOP/s), 15.7-17.4 against
// 18.6-19.7 with the fused pool; feature extraction 7 759 -> 8 017 images/s.  The dgrad launches (ReLU-mask strip, fused Gram block)
// are still slower than conv_c64 (25-28 against 21-24 us) and stay there.  Two things made the forward win: (i) the cut points of
// the CTAs' shares are KERNEL PARAMETERS -- with loop bounds that come out of in-kernel divisions ptxas keeps the descriptor words
// in vector registers and wraps every tcgen05.mma in an ELECT / R2UR.BROADCAST loop (14 SASS instructions per MMA, ~80 cycles);
// with uniform bounds and the eight-strip straight-line steady state it is 10 --, (ii) probes of the next strip's barriers are
// issued before the current strip's MMAs.  What bounds it now is shared-memory bandwidth: operands (120 KB per strip), patch,
// staging tile and TMA store come to ~190 KB per 128 pixels at 128 B/clk.
#include <algorithm>

#include "isx_common.cuh"
#include "isx_internal.h"
#include "isx_kernels.h"

namespace isx {

static constexpr int kSwThreads = 64 + 256;
static constexpr int kSwPatch = 17 * 1024;    // one strip patch: 130 rows x 128 B = 16640 B, padded to a multiple of 1024
static constexpr int kSwPatchBytes = 130 * 128;
static constexpr int kSwTile = 128 * 128;     // a 128-row x 64-channel bf16 tile
static constexpr int kSwWBytes = 9 * 64 * 128;  // nine 64 x 64 weight slabs
static constexpr int kSwMaxCtas = 160;          // persistent CTAs (one per SM; B200: 148)

struct SweepParams {
  int B, H, W;
  int U, V;            // extents of the strip axis and of the sweep axis
  int u_is_y;          // 1: strips run along y (u = y, v = x); 0: along x
  int u_tiles;         // strip positions per image
  long total_cols;     // B * u_tiles * V output strips in all
  // cut points of the CTAs' shares, computed by the host: share c = [cut c, cut c+1), a cut = (image, strip position, even v).
  // Kernel PARAMETERS on purpose: loop bounds read from the constant bank with a uniform index keep the whole issue loop in
  // uniform registers (with bounds derived by 64-bit divisions in the kernel, ptxas keeps the descriptor words in vector
  // registers and wraps every tcgen05.mma in two more instructions).
  int cut_b[kSwMaxCtas + 1], cut_t[kSwMaxCtas + 1], cut_v[kSwMaxCtas + 1];
  int patch_slots;
  int relu, fuse_pool, use_mask, use_gram, skip_out;
  const float* bias;
  const __nv_bfloat16* add_buf;
  const float* aff_a;
  const float* aff_b;
  uint8_t* pool_idx;
};

struct SweepLayout {
  int w, d, patch, act, stg, pstg, bars, total;
};
__host__ __device__ inline SweepLayout sweep_layout(int patch_slots, int use_mask, int use_gram, int fuse_pool) {
  SweepLayout L;
  int off = 0;
  L.w = off; off += kSwWBytes;
  L.d = off; off += use_gram ? 2 * 8192 : 0;
  L.patch = off; off += patch_slots * kSwPatch;
  // dgrad: FOUR ReLU-mask strips in flight (with two, the next strip's activation is requested only ~1.5 strip times before it
  // is needed -- less than a DRAM round trip: the epilogue then waited ~1 400 cycles per strip for it); the result is written
  // IN PLACE over the mask strip it was computed from, so the dgrad needs no staging tiles
  L.act = off; off += use_mask ? 4 * kSwTile : 0;
  L.stg = off; off += use_mask ? 0 : 2 * kSwTile;
  L.pstg = off; off += fuse_pool ? 2 * 8192 : 0;
  L.bars = off; off += 1024;
  L.total = off;
  return L;
}

// The output strips of the whole launch form one sequence f = (image b, strip position t, sweep coordinate v), v fastest.  CTA c
// owns the contiguous range [cut(c), cut(c + 1)) -- equal shares, cut at even v so that the pooling pairs stay together --
// and walks it as JOBS: maximal runs [vs, ve] inside one sweep (b, t).  Where a run starts or ends inside a sweep the
// neighbouring input strip is read as a halo; at the ends of a sweep the image border supplies zeros.
struct SweepJob {
  int b, u0, vs, ve, vin0, vin1;
};
struct SweepWalk {
  int b, t, v, b_end, t_end, v_end, V, u_tiles;
  __device__ SweepWalk(const SweepParams& p) : V(p.V), u_tiles(p.u_tiles) {
    const int c = blockIdx.x;
    b = p.cut_b[c]; t = p.cut_t[c]; v = p.cut_v[c];
    b_end = p.cut_b[c + 1]; t_end = p.cut_t[c + 1]; v_end = p.cut_v[c + 1];
  }
  __device__ bool next(SweepJob& J) {
    const bool last = b == b_end && t == t_end;
    if (last && v >= v_end) return false;
    J.vs = v;
    J.ve = (last ? v_end : V) - 1;
    J.b = b;
    J.u0 = t * 128;
    J.vin0 = max(J.vs - 1, 0);          // first / last input strip that contributes to the run
    J.vin1 = min(J.ve + 1, V - 1);
    if (last) {
      v = v_end;
    } else {
      v = 0;
      if (++t == u_tiles) { t = 0; ++b; }
    }
    return true;
  }
};

// The MMAs of one INTERIOR input strip (all three outputs exist, none of them is new except j = 2) whose output j = 0 sits in
// ring slot S: every TMEM address, instruction descriptor and accumulate flag is a compile-time constant, the shared-memory
// descriptors are the strip's base words plus immediates.  Twelve (ku, k) steps; the window (S, S+1, S+2) is one N = 192 MMA
// unless it wraps around the ring (S = 6, 7: two MMAs); the first step gives the new slot j = 2 its own MMA with accumulate = 0.
// uz: a runtime value that is always zero, derived from a kernel parameter -- added to the constant TMEM addresses so that
// they are formed on the uniform datapath (a literal goes through a vector register and an R2UR per MMA).
template <int S>
__device__ __forceinline__ void sweep_interior(uint32_t a_lo, uint32_t w_lo, uint32_t hi, uint32_t uz) {
  constexpr uint32_t I64 = umma_idesc_bf16(128, 64, false, false);
  constexpr uint32_t I128 = umma_idesc_bf16(128, 128, false, false);
  constexpr uint32_t I192 = umma_idesc_bf16(128, 192, false, false);
  constexpr uint32_t J1 = 8192 >> 4, J2 = 16384 >> 4;   // weight slab of output j inside the strip-tap block
#pragma unroll
  for (int ku = 0; ku < 3; ++ku) {
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const uint32_t a = a_lo + ((ku * 128 + k * 32) >> 4);
      const uint32_t b = w_lo + ((ku * 3 * 8192 + k * 32) >> 4);
      if (ku == 0 && k == 0) {
        if (S <= 6) {
          umma_bf16_lohi(S * 64 + uz, a, hi, b, hi, I128, 1u);
        } else {
          umma_bf16_lohi(448 + uz, a, hi, b, hi, I64, 1u);
          umma_bf16_lohi(uz, a, hi, b + J1, hi, I64, 1u);
        }
        umma_bf16_lohi(((S + 2) & 7) * 64 + uz, a, hi, b + J2, hi, I64, 0u);
      } else if (S <= 5) {
        umma_bf16_lohi(S * 64 + uz, a, hi, b, hi, I192, 1u);
      } else if (S == 6) {
        umma_bf16_lohi(384 + uz, a, hi, b, hi, I128, 1u);
        umma_bf16_lohi(uz, a, hi, b + J2, hi, I64, 1u);
      } else {
        umma_bf16_lohi(448 + uz, a, hi, b, hi, I64, 1u);
        umma_bf16_lohi(uz, a, hi, b + J1, hi, I128, 1u);
      }
    }
  }
}
// fused Gram backward of one output strip in ring slot S: + act . D_b (N = 64, K = 64)
template <int S>
__device__ __forceinline__ void sweep_gram(uint32_t a2, uint32_t b2, uint32_t hi) {
  constexpr uint32_t I64 = umma_idesc_bf16(128, 64, false, false);
#pragma unroll
  for (int k = 0; k < 4; ++k) umma_bf16_lohi(S * 64, a2 + 2 * k, hi, b2 + 2 * k, hi, I64, 1u);
}
#define ISX_SWEEP_SWITCH(slot, CALL)                 \
  switch (slot) {                                    \
    case 0: CALL(0); break; case 1: CALL(1); break;  \
    case 2: CALL(2); break; case 3: CALL(3); break;  \
    case 4: CALL(4); break; case 5: CALL(5); break;  \
    case 6: CALL(6); break; default: CALL(7); break; \
  }

__global__ void __launch_bounds__(kSwThreads, 1)
conv_sweep64_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmW,
                    const __grid_constant__ CUtensorMap tmO, const __grid_constant__ CUtensorMap tmM,
                    const __grid_constant__ CUtensorMap tmD, const __grid_constant__ CUtensorMap tmP, const SweepParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const SweepLayout L = sweep_layout(p.patch_slots, p.use_mask, p.use_gram, p.fuse_pool);
  const int PS = p.patch_slots;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + L.bars);
  uint64_t* w_full = bars;               // [1]
  uint64_t* patch_full = bars + 1;       // [8]
  uint64_t* patch_empty = bars + 9;      // [8]
  uint64_t* act_full = bars + 17;        // [4]
  uint64_t* act_empty = bars + 21;       // [4]
  uint64_t* d_full = bars + 25;          // [2]
  uint64_t* d_empty = bars + 27;         // [2]
  uint64_t* slot_full = bars + 29;       // [8]
  uint64_t* slot_empty = bars + 37;      // [8]
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(bars + 45);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmW);
    tma_prefetch_desc(&tmO);
    if (p.use_mask) tma_prefetch_desc(&tmM);
    if (p.use_gram) tma_prefetch_desc(&tmD);
    if (p.fuse_pool) tma_prefetch_desc(&tmP);
    mbar_init(w_full, 1);
    for (int i = 0; i < 8; ++i) {
      mbar_init(&patch_full[i], 1);
      mbar_init(&patch_empty[i], 1);
      mbar_init(&slot_full[i], 1);
      mbar_init(&slot_empty[i], 8);   // one arrival per epilogue warp
    }
    for (int i = 0; i < 4; ++i) {
      mbar_init(&act_full[i], 1);
      mbar_init(&act_empty[i], 1);    // the epilogue leader, once the TMA store of the result written over the strip has read it
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&d_full[i], 1);
      mbar_init(&d_empty[i], 1);
    }
    fence_barrier_init();
  }
  // the accumulator ring IS the whole tensor memory of the SM (see conv_c64.cu: base 0 by construction)
  if (warp == 1) tmem_alloc<512>(tmem_ptr_smem);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;

  if (warp == 0) {
    // ================================ TMA producer =========================================
    if (lane == 0) {
      // weight slab of strip tap ku: [j = 0..2][64 output channels][64 input channels], j <-> sweep tap ks = 2 - j
      mbar_arrive_expect_tx(w_full, kSwWBytes);
      for (int ky = 0; ky < 3; ++ky)
        for (int kx = 0; kx < 3; ++kx) {
          const int ku = p.u_is_y ? ky : kx, ks = p.u_is_y ? kx : ky;
          tma_load_2d(smem + L.w + (ku * 3 + (2 - ks)) * 8192, &tmW, w_full, 0, (ky * 3 + kx) * 64);
        }
      uint32_t ps = 0, pph = 0, as = 0, aph = 0, ds = 0, dph = 0;
      auto load_act = [&](int u0, int vo, int b) {
        mbar_wait(&act_empty[as], aph ^ 1);
        mbar_arrive_expect_tx(&act_full[as], kSwTile);
        tma_load_4d(smem + L.act + as * kSwTile, &tmM, &act_full[as], 0, u0, vo, b);
        if (++as == 4) { as = 0; aph ^= 1; }
      };
      SweepWalk walk(p);
      SweepJob J;
      while (walk.next(J)) {
        if (p.use_gram) {
          mbar_wait(&d_empty[ds], dph ^ 1);
          mbar_arrive_expect_tx(&d_full[ds], 8192);
          tma_load_2d(smem + L.d + ds * 8192, &tmD, &d_full[ds], 0, J.b * 64);
          ds ^= 1;
          if (ds == 0) dph ^= 1;
        }
        for (int vin = J.vin0; vin <= J.vin1; ++vin) {
          mbar_wait(&patch_empty[ps], pph ^ 1);
          mbar_arrive_expect_tx(&patch_full[ps], kSwPatchBytes);
          tma_load_4d(smem + L.patch + ps * kSwPatch, &tmA, &patch_full[ps], 0, J.u0 - 1, vin, J.b);
          if (++ps == static_cast<uint32_t>(PS)) { ps = 0; pph ^= 1; }
          if (p.use_mask) {  // activation strips of the outputs this input strip completes, in completion order
            if (vin - 1 >= J.vs) load_act(J.u0, vin - 1, J.b);
            if (vin == J.vin1 && vin <= J.ve) load_act(J.u0, vin, J.b);
          }
        }
      }
    }
  } else if (warp == 1) {
    // ================================ MMA issuer ===========================================
    if (lane == 0) {
      if (tmem_base != 0) {
        printf("isx: unexpected TMEM base %u (block %d)\n", tmem_base, blockIdx.x);
        __trap();
      }
      constexpr uint32_t idesc64 = umma_idesc_bf16(128, 64, false, false);
      constexpr uint32_t idesc_step = (64u >> 3) << 17;   // + one 64-column block of N
      mbar_wait(w_full, 0);
      const uint64_t dw0 = umma_desc_sw128(smem_u32(smem + L.w), 16, 1024);
      const uint64_t da0 = umma_desc_sw128(smem_u32(smem + L.patch), 16, 1024);
      const uint32_t w_lo = static_cast<uint32_t>(dw0), hi = static_cast<uint32_t>(dw0 >> 32);  // same high word everywhere
      const uint32_t a_lo0 = static_cast<uint32_t>(da0);
      const uint32_t act_lo0 = static_cast<uint32_t>(umma_desc_sw128(smem_u32(smem + L.act), 16, 1024));
      const uint32_t d_lo0 = static_cast<uint32_t>(umma_desc_sw128(smem_u32(smem + L.d), 16, 1024));
      const uint32_t uz = p.B < 0 ? 64u : 0u;   // always 0, but only the hardware knows
      uint32_t ps = 0, pph = 0, as = 0, aph = 0, a_lo = a_lo0;
      bool p_ready = false, s_ready = false, a_ready = false;
      uint32_t s_probed = 0xffffffffu;
      uint32_t ds = 0, dph = 0;
      uint32_t g0 = 0;           // running number of the job's first output strip
      // An mbarrier probe costs 150-270 cycles even when its phase completed long ago: the probes of the NEXT strip's
      // barriers (its patch, the ring slot it touches first) are issued before this strip's MMAs and consumed afterwards.
      SweepWalk walk(p);
      SweepJob J;
      while (walk.next(J)) {
        if (p.use_gram) mbar_wait(&d_full[ds], dph);
        for (int vin = J.vin0; vin <= J.vin1; ++vin) {
          const int ja = max(0, J.vs - vin + 1), jb = min(2, J.ve - vin + 1);   // valid outputs vo = vin - 1 + j
          const uint32_t gj0 = g0 + static_cast<uint32_t>(vin - 1 - J.vs);      // running number of output j = 0 (may be "-1")
          const bool first_in = vin == J.vin0;
          // steady state: eight interior strips in a row, starting ring-aligned -> straight-line code with constant slots
          if ((gj0 & 7) == 0 && !first_in && vin - 1 >= J.vs && vin + 8 <= J.ve) {
            const uint32_t q = (gj0 >> 3) & 1;
            const uint32_t d_lo = d_lo0 + ds * (8192 >> 4);
#define ISX_SWEEP_FAST(S_)                                                                                                   \
  {                                                                                                                          \
    if (!(s_ready && s_probed == gj0 + S_ + 2)) mbar_wait(&slot_empty[(S_ + 2) & 7], q ^ (S_ >= 6 ? 1u : 0u) ^ 1u);           \
    if (!p_ready) mbar_wait(&patch_full[ps], pph);                                                                           \
    tc_fence_after();                                                                                                        \
    {                                                                                                                        \
      const uint32_t ps_n = ps + 1 == static_cast<uint32_t>(PS) ? 0 : ps + 1;                                                \
      p_ready = mbar_try_wait(&patch_full[ps_n], ps_n == 0 ? pph ^ 1 : pph);                                                 \
      s_probed = gj0 + S_ + 3;                                                                                               \
      s_ready = mbar_try_wait(&slot_empty[(S_ + 3) & 7], q ^ (S_ >= 5 ? 1u : 0u) ^ 1u);                                       \
      if (p.use_gram) a_ready = mbar_try_wait(&act_full[as], aph);                                                           \
    }                                                                                                                        \
    sweep_interior<S_>(a_lo, w_lo, hi, uz);                                                                                      \
    umma_commit(&patch_empty[ps]);                                                                                           \
    a_lo += kSwPatch >> 4;                                                                                                   \
    if (++ps == static_cast<uint32_t>(PS)) { ps = 0; pph ^= 1; a_lo = a_lo0; }                                               \
    if (p.use_gram) {                                                                                                        \
      if (!a_ready) mbar_wait(&act_full[as], aph);                                                                           \
      tc_fence_after();                                                                                                      \
      sweep_gram<S_>(act_lo0 + as * (kSwTile >> 4), d_lo, hi);                                                               \
      if (++as == 4) { as = 0; aph ^= 1; }                                                                                   \
    }                                                                                                                        \
    umma_commit(&slot_full[S_]);                                                                                             \
  }
            ISX_SWEEP_FAST(0); ISX_SWEEP_FAST(1); ISX_SWEEP_FAST(2); ISX_SWEEP_FAST(3);
            ISX_SWEEP_FAST(4); ISX_SWEEP_FAST(5); ISX_SWEEP_FAST(6); ISX_SWEEP_FAST(7);
#undef ISX_SWEEP_FAST
            vin += 7;
            continue;
          }
          const bool interior = !first_in && ja == 0 && jb == 2;
          // first touches (in running order): everything at the first input strip of a job, afterwards only j = 2
          for (int j = first_in ? ja : 2; j <= jb; ++j) {
            const uint32_t g = gj0 + j;
            if (!(s_ready && s_probed == g)) mbar_wait(&slot_empty[g & 7], ((g >> 3) & 1) ^ 1);
          }
          if (!p_ready) mbar_wait(&patch_full[ps], pph);
          tc_fence_after();
          {
            const uint32_t ps_n = ps + 1 == static_cast<uint32_t>(PS) ? 0 : ps + 1;
            p_ready = mbar_try_wait(&patch_full[ps_n], ps_n == 0 ? pph ^ 1 : pph);
            s_probed = gj0 + 3;   // the slot the next strip touches first (when it is an ordinary strip)
            s_ready = mbar_try_wait(&slot_empty[s_probed & 7], ((s_probed >> 3) & 1) ^ 1);
          }
          if (interior) {
#define ISX_SWEEP_CALL(S_) sweep_interior<S_>(a_lo, w_lo, hi, uz)
            ISX_SWEEP_SWITCH(gj0 & 7, ISX_SWEEP_CALL)
#undef ISX_SWEEP_CALL
          } else {
            // edge strips of a job (two at each end): the MMAs of one (ku, k) step for outputs j0..j1, consecutive ring slots,
            // split where the ring wraps
            auto emit = [&](int j0, int j1, uint32_t a_desc, uint32_t b_desc, uint32_t accum) {
              const uint32_t s0 = (gj0 + j0) & 7;
              const int n = j1 - j0 + 1;
              const int n1 = min(n, 8 - static_cast<int>(s0));
              umma_bf16_lohi(s0 * 64, a_desc, hi, b_desc + ((j0 * 8192) >> 4), hi, idesc64 + (n1 - 1) * idesc_step, accum);
              if (n1 < n)
                umma_bf16_lohi(0, a_desc, hi, b_desc + (((j0 + n1) * 8192) >> 4), hi, idesc64 + (n - n1 - 1) * idesc_step, accum);
            };
#pragma unroll
            for (int ku = 0; ku < 3; ++ku) {
#pragma unroll
              for (int k = 0; k < 4; ++k) {
                const uint32_t a_desc = a_lo + ((ku * 128 + k * 32) >> 4);
                const uint32_t b_desc = w_lo + ((ku * 3 * 8192 + k * 32) >> 4);
                if (ku == 0 && k == 0) {
                  if (first_in) {
                    emit(ja, jb, a_desc, b_desc, 0u);
                  } else {
                    if (ja <= min(jb, 1)) emit(ja, min(jb, 1), a_desc, b_desc, 1u);
                    if (jb == 2) emit(2, 2, a_desc, b_desc, 0u);
                  }
                } else {
                  emit(ja, jb, a_desc, b_desc, 1u);
                }
              }
            }
          }
          umma_commit(&patch_empty[ps]);
          a_lo += kSwPatch >> 4;
          if (++ps == static_cast<uint32_t>(PS)) { ps = 0; pph ^= 1; a_lo = a_lo0; }
          // outputs that are complete now: vin - 1, and vin itself at the last input strip of a run that ends at the image border
          for (int c = 0; c < 2; ++c) {
            const int vo = c == 0 ? vin - 1 : vin;
            if (c == 0 ? (vo < J.vs) : !(vin == J.vin1 && vin <= J.ve)) continue;
            const uint32_t g = g0 + static_cast<uint32_t>(vo - J.vs);
            if (p.use_gram) {
              mbar_wait(&act_full[as], aph);
              tc_fence_after();
              const uint32_t a2 = act_lo0 + as * (kSwTile >> 4), b2 = d_lo0 + ds * (8192 >> 4);
#define ISX_SWEEP_CALL(S_) sweep_gram<S_>(a2, b2, hi)
              ISX_SWEEP_SWITCH(g & 7, ISX_SWEEP_CALL)
#undef ISX_SWEEP_CALL
              if (++as == 4) { as = 0; aph ^= 1; }
            }
            umma_commit(&slot_full[g & 7]);
          }
        }
        if (p.use_gram) {
          umma_commit(&d_empty[ds]);
          ds ^= 1;
          if (ds == 0) dph ^= 1;
        }
        g0 += static_cast<uint32_t>(J.ve - J.vs + 1);
      }
    }
  } else {
    // ================================ epilogue (8 warps) ===================================
    const int q = warp & 3;
    const int hsel = (warp - 2) >> 2;
    const int row = q * 32 + lane;
    const int n = hsel * 32;            // this thread's 32 output channels
    const bool leader = threadIdx.x == 64;
    float bias_r[32];
#pragma unroll
    for (int e = 0; e < 32; ++e) bias_r[e] = p.bias != nullptr ? __ldg(p.bias + n + e) : 0.f;
    uint32_t g = 0, at = 0;   // running output-strip / activation-strip counters
    uint32_t act_held = 0xffffffffu;   // leader: mask strip whose in-place result is still being read by its TMA store
    bool f_ready = false;     // slot_full of strip g already seen (probed while the previous strip was in flight)
    bool m_ready = false;     // likewise the ReLU-mask strip of strip g (dgrad)
    const bool regpool = p.fuse_pool && p.skip_out && !p.use_mask;   // pool in registers, nothing else to store
    uint32_t prevw[16];       // regpool: the even strip of the current pair, packed bf16x2
#pragma unroll
    for (int e = 0; e < 16; ++e) prevw[e] = 0u;
    SweepWalk walk(p);
    SweepJob J;
    while (walk.next(J)) {
      const int u = J.u0 + row;
      const bool valid = u < p.U;
      for (int vo = J.vs; vo <= J.ve; ++vo, ++g) {
        const uint32_t slot = g & 7;
        const int px = p.u_is_y ? vo : u, py = p.u_is_y ? u : vo;
        const size_t pix = valid ? ((static_cast<size_t>(J.b) * p.H + py) * p.W + px) * 64 : 0;
        const uint32_t ss = static_cast<uint32_t>(vo) & 1;   // staging slot: even / odd sweep coordinate
        const uint32_t as = at & 3;                          // dgrad: mask strip of this output, overwritten in place by the result
        uint8_t* stg = p.use_mask ? smem + L.act + as * kSwTile : smem + L.stg + ss * kSwTile;
        if (!f_ready) mbar_wait(&slot_full[slot], (g >> 3) & 1);
        tc_fence_after();
        uint32_t v[32];
        tmem_ld_32x32(tmem_base + slot * 64 + n + (static_cast<uint32_t>(q * 32) << 16), v);
        tmem_ld_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&slot_empty[slot]);   // accumulator read: the ring slot goes back to the MMA warp
        f_ready = mbar_try_wait(&slot_full[(g + 1) & 7], ((g + 1) >> 3) & 1);   // consumed at the top of the next strip
        const bool m_now = m_ready;
        if (p.use_mask) m_ready = mbar_try_wait(&act_full[(at + 1) & 3], ((at + 1) >> 2) & 1);
        float f[32];
#pragma unroll
        for (int e = 0; e < 32; ++e) f[e] = __uint_as_float(v[e]) + bias_r[e];
        if (p.add_buf != nullptr && valid) {
#pragma unroll
          for (int e = 0; e < 32; e += 8) {
            const uint4 w4 = __ldg(reinterpret_cast<const uint4*>(p.add_buf + pix + n + e));
            float2 t;
            t = unpack_bf16x2(w4.x); f[e] += t.x; f[e + 1] += t.y;
            t = unpack_bf16x2(w4.y); f[e + 2] += t.x; f[e + 3] += t.y;
            t = unpack_bf16x2(w4.z); f[e + 4] += t.x; f[e + 5] += t.y;
            t = unpack_bf16x2(w4.w); f[e + 6] += t.x; f[e + 7] += t.y;
          }
        }
        // ReLU mask of the layer below as packed select masks (0xFFFF per bf16 whose activation is > 0): applied to the packed
        // output words -- one HSETP2 + one AND per two channels instead of two unpacks and two selects
        uint32_t keep[16];
#pragma unroll
        for (int e = 0; e < 16; ++e) keep[e] = 0xffffffffu;
        if (p.use_mask) {
          if (!m_now) mbar_wait(&act_full[as], (at >> 2) & 1);
          const uint8_t* mrow = stg + row * 128;   // read before this thread overwrites the same 16-byte chunks below
          const __nv_bfloat162 zero2 = __floats2bfloat162_rn(0.f, 0.f);
#pragma unroll
          for (int e = 0; e < 32; e += 8) {
            const int chunk = (hsel * 4 + (e >> 3)) ^ (row & 7);
            const uint4 w4 = *reinterpret_cast<const uint4*>(mrow + chunk * 16);
            const uint32_t ww[4] = {w4.x, w4.y, w4.z, w4.w};
#pragma unroll
            for (int i = 0; i < 4; ++i) keep[(e >> 1) + i] = __hgt2_mask(*reinterpret_cast<const __nv_bfloat162*>(&ww[i]), zero2);
            if (p.aff_a != nullptr && valid) {
              float a[8];
              float2 t;
              t = unpack_bf16x2(w4.x); a[0] = t.x; a[1] = t.y;
              t = unpack_bf16x2(w4.y); a[2] = t.x; a[3] = t.y;
              t = unpack_bf16x2(w4.z); a[4] = t.x; a[5] = t.y;
              t = unpack_bf16x2(w4.w); a[6] = t.x; a[7] = t.y;
              const float* pa = p.aff_a + static_cast<size_t>(J.b) * 64 + n + e;
              const float* pb = p.aff_b + static_cast<size_t>(J.b) * 64 + n + e;
#pragma unroll
              for (int j = 0; j < 8; ++j) f[e + j] += __ldg(pa + j) + __ldg(pb + j) * a[j];
            }
          }
          ++at;
        }
        if (p.relu) {
#pragma unroll
          for (int e = 0; e < 32; ++e) f[e] = fmaxf(f[e], 0.f);
        }
        if (regpool) {
          // Forward with the fused pool and NO full-resolution store (NST evaluation, lean feature forward): the 2x2 windows are
          // pooled IN REGISTERS.  The two strips of a window are consecutive strips of the same thread (the even one is kept in
          // prevw), its two rows are the lanes l and l ^ 1 of one warp.  No staging tile, no barrier on even strips, 32 KB less
          // shared-memory traffic per pair of strips -- the kernel's bound.
          uint32_t w[16];
#pragma unroll
          for (int e = 0; e < 16; ++e) w[e] = pack_bf16x2(f[2 * e], f[2 * e + 1]);
          if ((vo & 1) == 0) {
#pragma unroll
            for (int e = 0; e < 16; ++e) prevw[e] = w[e];
            continue;
          }
          const bool odd = (lane & 1) != 0;   // this lane pools words 8..15 of its 16, the even lane of the pair words 0..7
          uint32_t r0p[8], r1p[8], r0c[8], r1c[8];   // rows r0 (even lane) / r1 (odd lane) x strips prev / cur, this lane's 8 words
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const uint32_t my_p = odd ? prevw[8 + i] : prevw[i], send_p = odd ? prevw[i] : prevw[8 + i];
            const uint32_t my_c = odd ? w[8 + i] : w[i], send_c = odd ? w[i] : w[8 + i];
            const uint32_t got_p = __shfl_xor_sync(0xffffffffu, send_p, 1);
            const uint32_t got_c = __shfl_xor_sync(0xffffffffu, send_c, 1);
            r0p[i] = odd ? got_p : my_p; r1p[i] = odd ? my_p : got_p;
            r0c[i] = odd ? got_c : my_c; r1c[i] = odd ? my_c : got_c;
          }
          uint8_t* pst = smem + L.pstg + ((static_cast<uint32_t>(vo) >> 1) & 1) * 8192;
          const int pr = row >> 1;
          const int up = (J.u0 >> 1) + pr, vp = vo >> 1;
          const int xp = p.u_is_y ? vp : up, yp = p.u_is_y ? up : vp;
          const bool pvalid = xp < (p.W >> 1) && yp < (p.H >> 1);
          uint32_t cw[4];
#pragma unroll
          for (int h2 = 0; h2 < 2; ++h2) {
            uint4 u4[4];
            // window scan order (dy, dx): u = y -> (r0,prev) (r0,cur) (r1,prev) (r1,cur); u = x -> (prev,r0) (prev,r1) (cur,r0) (cur,r1)
            u4[0] = make_uint4(r0p[4 * h2], r0p[4 * h2 + 1], r0p[4 * h2 + 2], r0p[4 * h2 + 3]);
            u4[3] = make_uint4(r1c[4 * h2], r1c[4 * h2 + 1], r1c[4 * h2 + 2], r1c[4 * h2 + 3]);
            const uint4 a = make_uint4(r0c[4 * h2], r0c[4 * h2 + 1], r0c[4 * h2 + 2], r0c[4 * h2 + 3]);
            const uint4 bq = make_uint4(r1p[4 * h2], r1p[4 * h2 + 1], r1p[4 * h2 + 2], r1p[4 * h2 + 3]);
            u4[1] = p.u_is_y ? a : bq;
            u4[2] = p.u_is_y ? bq : a;
            uint4 m4;
            uint2 codes;
            pool4_codes(u4, m4, codes);
            cw[2 * h2] = codes.x; cw[2 * h2 + 1] = codes.y;
            const int chunk = hsel * 4 + (odd ? 2 : 0) + h2;   // 16-byte chunk (8 channels) of the pooled row
            *reinterpret_cast<uint4*>(pst + pr * 128 + ((chunk ^ (pr & 7)) * 16)) = m4;
          }
          if (p.pool_idx != nullptr && pvalid)
            *reinterpret_cast<uint4*>(p.pool_idx + ((static_cast<size_t>(J.b) * (p.H >> 1) + yp) * (p.W >> 1) + xp) * 64 + hsel * 32 +
                                      (odd ? 16 : 0)) = make_uint4(cw[0], cw[1], cw[2], cw[3]);
          fence_proxy_async_smem();
          if (leader) tma_store_wait_read<0>();   // the pooled tile written two pairs ago has been read by its store
          asm volatile("bar.sync 1, 256;" ::: "memory");
          if (leader) {
            tma_store_4d(&tmP, pst, 0, J.u0 >> 1, vo >> 1, J.b);
            tma_store_commit();
          }
          continue;
        }
        uint8_t* rowp = stg + row * 128;
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          uint4 o;
          o.x = pack_bf16x2(f[c * 8 + 0], f[c * 8 + 1]) & keep[c * 4 + 0];
          o.y = pack_bf16x2(f[c * 8 + 2], f[c * 8 + 3]) & keep[c * 4 + 1];
          o.z = pack_bf16x2(f[c * 8 + 4], f[c * 8 + 5]) & keep[c * 4 + 2];
          o.w = pack_bf16x2(f[c * 8 + 6], f[c * 8 + 7]) & keep[c * 4 + 3];
          const int chunk = (hsel * 4 + c) ^ (row & 7);
          *reinterpret_cast<uint4*>(rowp + chunk * 16) = o;
        }
        fence_proxy_async_smem();
        // the other staging slot is rewritten by the next strip: the TMA stores that read it must be done with it
        if (leader) {
          tma_store_wait_read<0>();
          if (act_held != 0xffffffffu) { mbar_arrive(&act_empty[act_held]); act_held = 0xffffffffu; }   // its store has read it
        }
        asm volatile("bar.sync 1, 256;" ::: "memory");
        if (leader && !p.skip_out) {
          tma_store_4d(&tmO, stg, 0, J.u0, vo, J.b);
          tma_store_commit();
        }
        if (leader && p.use_mask) act_held = as;
        if (p.fuse_pool && (vo & 1)) {
          // 2x2 max-pool of strips vo - 1 (staging slot 0) and vo (slot 1): 64 pooled pixels x 64 channels, 2 items per thread
          const uint8_t* s0 = smem + L.stg;
          const uint8_t* s1 = smem + L.stg + kSwTile;
          uint8_t* pst = smem + L.pstg + ((static_cast<uint32_t>(vo) >> 1) & 1) * 8192;
#pragma unroll
          for (int rep = 0; rep < 2; ++rep) {
            const int item = static_cast<int>(threadIdx.x) - 64 + rep * 256;   // 0..511
            const int pr = item >> 3, chunk = item & 7;
            const int r0 = 2 * pr, r1 = 2 * pr + 1;
            const int o0 = r0 * 128 + ((chunk ^ (r0 & 7)) * 16), o1 = r1 * 128 + ((chunk ^ (r1 & 7)) * 16);
            uint4 u4[4];
            // window scan order (dy, dx): u = y -> (r0,s0) (r0,s1) (r1,s0) (r1,s1); u = x -> (s0,r0) (s0,r1) (s1,r0) (s1,r1)
            u4[0] = *reinterpret_cast<const uint4*>(s0 + o0);
            u4[3] = *reinterpret_cast<const uint4*>(s1 + o1);
            if (p.u_is_y) {
              u4[1] = *reinterpret_cast<const uint4*>(s1 + o0);
              u4[2] = *reinterpret_cast<const uint4*>(s0 + o1);
            } else {
              u4[1] = *reinterpret_cast<const uint4*>(s0 + o1);
              u4[2] = *reinterpret_cast<const uint4*>(s1 + o0);
            }
            uint4 m4;
            uint2 codes;
            pool4_codes(u4, m4, codes);
            if (p.pool_idx != nullptr) {
              const int up = (J.u0 >> 1) + pr, vp = vo >> 1;
              const int xp = p.u_is_y ? vp : up, yp = p.u_is_y ? up : vp;
              if (xp < (p.W >> 1) && yp < (p.H >> 1))
                *reinterpret_cast<uint2*>(p.pool_idx + ((static_cast<size_t>(J.b) * (p.H >> 1) + yp) * (p.W >> 1) + xp) * 64 +
                                          chunk * 8) = codes;
            }
            *reinterpret_cast<uint4*>(pst + pr * 128 + ((chunk ^ (pr & 7)) * 16)) = m4;
          }
          fence_proxy_async_smem();
          asm volatile("bar.sync 1, 256;" ::: "memory");
          if (leader) {
            tma_store_4d(&tmP, pst, 0, J.u0 >> 1, vo >> 1, J.b);
            tma_store_commit();
          }
        }
      }
    }
    if (leader) {
      tma_store_wait_all<0>();
      if (act_held != 0xffffffffu) mbar_arrive(&act_empty[act_held]);
    }
    tc_fence_before();
  }
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc<512>(tmem_base);
  }
}

// fraction of the 128 strip positions that hold real pixels when the strip axis has `n` pixels
static double strip_efficiency(int n) { return static_cast<double>(n) / (((n + 127) / 128) * 128); }

bool conv_sweep_applicable(const ConvArgs& a) {
  if (a.Cin != 64 || a.Cout != 64 || a.ntaps != 9 || a.per_image_weights || a.dx_nchw != nullptr || a.stride != 1) return false;
  if (a.out == nullptr) return false;
  if (a.gram_act != nullptr && a.gram_act != a.mask_act) return false;
  if (a.aff_a != nullptr && a.mask_act == nullptr) return false;
  return true;
}
double conv_sweep_efficiency(const ConvArgs& a) { return std::max(strip_efficiency(a.H), strip_efficiency(a.W)); }

int conv_sweep(const ConvArgs& a, cudaStream_t stream) {
  ISX_REQUIRE(conv_sweep_applicable(a), "conv_sweep: not applicable");
  SweepParams p;
  memset(&p, 0, sizeof(p));
  p.B = a.B; p.H = a.H; p.W = a.W;
  // strip axis: the one that fills its 128-pixel strips better; ties go to x (contiguous strips)
  p.u_is_y = strip_efficiency(a.H) > strip_efficiency(a.W) ? 1 : 0;
  p.U = p.u_is_y ? a.H : a.W;
  p.V = p.u_is_y ? a.W : a.H;
  p.u_tiles = (p.U + 127) / 128;
  p.total_cols = static_cast<long>(a.B) * p.u_tiles * p.V;
  p.relu = a.relu; p.bias = a.bias; p.add_buf = a.add_buf; p.aff_a = a.aff_a; p.aff_b = a.aff_b;
  p.use_mask = a.mask_act != nullptr ? 1 : 0;
  p.use_gram = a.gram_act != nullptr ? 1 : 0;
  p.fuse_pool = (a.pool_out != nullptr && a.H >= 2 && a.W >= 2) ? 1 : 0;
  p.pool_idx = p.fuse_pool ? a.pool_idx : nullptr;
  p.skip_out = (p.fuse_pool && a.pool_idx != nullptr && a.skip_out) ? 1 : 0;
  int ps = 6;
  SweepLayout L = sweep_layout(ps, p.use_mask, p.use_gram, p.fuse_pool);
  while (ps > 2 && 1024 + L.total > 227 * 1024) { --ps; L = sweep_layout(ps, p.use_mask, p.use_gram, p.fuse_pool); }
  ISX_REQUIRE(1024 + L.total <= 227 * 1024, "conv_sweep: %d B of shared memory exceed 227 KB", 1024 + L.total);
  p.patch_slots = ps;
  const size_t smem_bytes = std::max<size_t>(1024 + L.total, 204 * 1024);  // nobody else of this library fits beside it

  // the NHWC tensors seen as (c, u, v, b): u = strip axis, v = sweep axis
  const uint64_t su = (p.u_is_y ? static_cast<uint64_t>(a.W) : 1ull) * 128, sv = (p.u_is_y ? 1ull : static_cast<uint64_t>(a.W)) * 128;
  const uint64_t sb = static_cast<uint64_t>(a.H) * a.W * 128;
  CUtensorMap tmA, tmW, tmO, tmM, tmD, tmP;
  {
    uint64_t dims[4] = {64, (uint64_t)p.U, (uint64_t)p.V, (uint64_t)a.B};
    uint64_t str[3] = {su, sv, sb};
    uint32_t box[4] = {64, 130, 1, 1};
    if (isx_make_tmap_bf16(&tmA, a.in, 4, dims, str, box, true)) return 3;
    uint32_t box2[4] = {64, 128, 1, 1};
    if (isx_make_tmap_bf16(&tmO, a.out, 4, dims, str, box2, true)) return 3;
    tmM = tmO;
    if (p.use_mask && isx_make_tmap_bf16(&tmM, a.mask_act, 4, dims, str, box2, true)) return 3;
  }
  {
    uint64_t dims[2] = {64, (uint64_t)9 * 64};
    uint64_t str[1] = {128};
    uint32_t box[2] = {64, 64};
    if (isx_make_tmap_bf16(&tmW, a.weight, 2, dims, str, box, true)) return 3;
  }
  tmD = tmW; tmP = tmO;
  if (p.use_gram) {
    uint64_t d2[2] = {64, (uint64_t)64 * a.B};
    uint64_t s2[1] = {128};
    uint32_t b2[2] = {64, 64};
    if (isx_make_tmap_bf16(&tmD, a.gram_D, 2, d2, s2, b2, true)) return 3;
  }
  if (p.fuse_pool) {
    const int Hp = a.H / 2, Wp = a.W / 2;
    uint64_t dp[4] = {64, (uint64_t)(p.u_is_y ? Hp : Wp), (uint64_t)(p.u_is_y ? Wp : Hp), (uint64_t)a.B};
    uint64_t sp[3] = {(p.u_is_y ? static_cast<uint64_t>(Wp) : 1ull) * 128, (p.u_is_y ? 1ull : static_cast<uint64_t>(Wp)) * 128,
                      static_cast<uint64_t>(Hp) * Wp * 128};
    uint32_t bp[4] = {64, 64, 1, 1};
    if (isx_make_tmap_bf16(&tmP, a.pool_out, 4, dp, sp, bp, true)) return 3;
  }
  ISX_CHECK_CUDA(cudaFuncSetAttribute(conv_sweep64_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bytes));
  // every CTA gets an equal contiguous share of the output strips; tiny launches: at least ~16 strips per CTA
  const long grid = std::max<long>(1, std::min<long>(p.total_cols / 16, std::min<long>(kNumSMs, kSwMaxCtas)));
  for (long k = 0; k <= grid; ++k) {
    long f = k >= grid ? p.total_cols : k * p.total_cols / grid;
    long sw = f / p.V;
    const long v = k >= grid ? 0 : ((f - sw * p.V) & ~1L);    // even v: the pooling pairs of strips stay in one share
    p.cut_b[k] = static_cast<int>(sw / p.u_tiles);
    p.cut_t[k] = static_cast<int>(sw % p.u_tiles);
    p.cut_v[k] = static_cast<int>(v);
  }
  isx_prof_begin(ISX_PROF_CONV, 2.0 * (9 * 64 + (p.use_gram ? 64 : 0)) * 64 * static_cast<double>(a.B) * a.H * a.W, stream);
  conv_sweep64_kernel<<<(unsigned)grid, kSwThreads, smem_bytes, stream>>>(tmA, tmW, tmO, tmM, tmD, tmP, p);
  isx_prof_end(ISX_PROF_CONV, stream);
  ISX_LAUNCH_CHECK();
  return 0;
}

}  // namespace isx
