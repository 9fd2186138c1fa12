// K7 / K8: torch.optim.LBFGS (no line search) as the reference uses it -- pipelines.py:59,103 ->
// torch/optim/lbfgs.py:333-537 -- re-designed for the device:
//
//  * P independent problems (one per image, SURVEY.md F6) advance in lock step, one closure
//    evaluation per "tick"; every scalar of the optimiser (loss, t, H_diag, ro, al, the early-exit
//    flags of lbfgs.py:370-374,463,511-526 and the 20-iterations-per-step bookkeeping) lives in a
//    per-problem device struct, so a tick needs no host synchronisation and can sit in a CUDA graph.
//  * The two-loop recursion (lbfgs.py:432-442: <=100 dot + <=100 axpy, twice, each a launch and a
//    pass over the parameter vector) is evaluated in COEFFICIENT SPACE.  With q = -g - sum_j al_j y_j
//    and r = gamma q + sum_j (al_j - be_j) s_j the recursion only needs the inner products s_i.g,
//    y_i.g, s_i.y_j, y_i.y_j; they are maintained incrementally (one new row per accepted pair), so
//    a tick streams the history twice in total:
//      pass 1 (lbfgs_dots):   y = g - g_prev (stored), all s_i.g, y_i.g, s_i.y, y_i.y, |g|_inf, |g|_1, g.g
//      control (lbfgs_control): state machine + O(m^2) scalar recursion -> coefficients, t, flags
//      pass 2 (lbfgs_update): d = cg g + sum cs_i s_i + cy_i y_i; s_new = t d (stored); g_prev = g;
//                             x = clamp(x + t d, 0, 1) (pipelines.py:82 fused: add -> clamp is the only
//                             order in which x is ever read); max|t d|
//    Mathematically identical to lbfgs.py:404-442; fp32 vectors, double scalars.
#include <algorithm>

#include "isx_common.cuh"
#include "isx_kernels.h"
#include "lbfgs_state.h"

namespace isx {

static constexpr int kDotThreads = 256;
static constexpr int kElemsPerThread = 8;
static constexpr int kChunk = kDotThreads * kElemsPerThread;  // elements per block

__host__ __device__ __forceinline__ int nblk_of(long N) { return static_cast<int>((N + kChunk - 1) / kChunk); }

__device__ __forceinline__ void load8(const float* p, long i, long n, float (&v)[8]) {
  if (i + 8 <= n && (reinterpret_cast<uintptr_t>(p + i) & 15) == 0) {
    const float4 a = __ldg(reinterpret_cast<const float4*>(p + i));
    const float4 b = __ldg(reinterpret_cast<const float4*>(p + i + 4));
    v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
  } else {
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] = (i + j < n) ? p[i + j] : 0.f;
  }
}
__device__ __forceinline__ void store8(float* p, long i, long n, const float (&v)[8]) {
  if (i + 8 <= n && (reinterpret_cast<uintptr_t>(p + i) & 15) == 0) {
    *reinterpret_cast<float4*>(p + i) = make_float4(v[0], v[1], v[2], v[3]);
    *reinterpret_cast<float4*>(p + i + 4) = make_float4(v[4], v[5], v[6], v[7]);
  } else {
#pragma unroll
    for (int j = 0; j < 8; ++j)
      if (i + j < n) p[i + j] = v[j];
  }
}

// history element type: float (the reference's fp32 state) or bf16 (opt-in: halves the HBM traffic of both passes)
__device__ __forceinline__ void hload8(const float* p, long i, long n, float (&v)[8]) { load8(p, i, n, v); }
__device__ __forceinline__ void hstore8(float* p, long i, long n, const float (&v)[8]) { store8(p, i, n, v); }
__device__ __forceinline__ void hload8(const __nv_bfloat16* p, long i, long n, float (&v)[8]) {
  if (i + 8 <= n && (reinterpret_cast<uintptr_t>(p + i) & 15) == 0) {
    const uint4 u = __ldg(reinterpret_cast<const uint4*>(p + i));
    float2 t;
    t = unpack_bf16x2(u.x); v[0] = t.x; v[1] = t.y;
    t = unpack_bf16x2(u.y); v[2] = t.x; v[3] = t.y;
    t = unpack_bf16x2(u.z); v[4] = t.x; v[5] = t.y;
    t = unpack_bf16x2(u.w); v[6] = t.x; v[7] = t.y;
  } else {
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] = (i + j < n) ? __bfloat162float(p[i + j]) : 0.f;
  }
}
__device__ __forceinline__ void hstore8(__nv_bfloat16* p, long i, long n, const float (&v)[8]) {
  if (i + 8 <= n && (reinterpret_cast<uintptr_t>(p + i) & 15) == 0) {
    uint4 u;
    u.x = pack_bf16x2(v[0], v[1]); u.y = pack_bf16x2(v[2], v[3]);
    u.z = pack_bf16x2(v[4], v[5]); u.w = pack_bf16x2(v[6], v[7]);
    *reinterpret_cast<uint4*>(p + i) = u;
  } else {
#pragma unroll
    for (int j = 0; j < 8; ++j)
      if (i + j < n) p[i + j] = __float2bfloat16_rn(v[j]);
  }
}
// what the stored (possibly rounded) value reads back as: the inner products must see exactly the stored pair
__device__ __forceinline__ float hround(float v, const float*) { return v; }
__device__ __forceinline__ float hround(float v, const __nv_bfloat16*) { return __bfloat162float(__float2bfloat16_rn(v)); }

// ---------------------------------------------------------------------------------------------
// pass 1
// partial layout: part[p][blk][slot][4] floats then extras: ext[p][blk][4] = {sum g^2, sum |g|, max |g|, 0}
// kPerProblem: problem p owns the floats [vb, vb + N_p) of g / g_prev / x (vb = pr.vec_begin(p), N_p = pr.vec_size(p)) and
// the history block S / Y + M1 * vb, slot k at k * N_p; the grid spans the largest problem (nblk blocks) and the blocks
// past lbfgs_nblk(N_p) return at once, so a problem's block partition, and with it its summation order, depends on N_p only
// ---------------------------------------------------------------------------------------------
template <typename HT, bool kPerProblem>
__global__ void __launch_bounds__(kDotThreads)
lbfgs_dots_kernel(const float* __restrict__ g, const float* __restrict__ g_prev, const HT* __restrict__ S,
                  HT* __restrict__ Y, const LbfgsState* __restrict__ states, long N, int M1, int nblk,
                  float* __restrict__ part, float* __restrict__ ext,
                  const __grid_constant__ ProblemArg<kPerProblem, ProblemRanges> pr) {
  const int p = blockIdx.y;
  const LbfgsState& st = states[p];
  if (st.done) return;
  long vb;
  if constexpr (kPerProblem) {
    vb = pr.vec_begin(p);
    N = pr.vec_size(p);
    if (static_cast<int>(blockIdx.x) >= nblk_of(N)) return;
  }
  // history slot k of problem p
  auto hist = [&](int k) -> long {
    if constexpr (kPerProblem) return M1 * vb + k * N;
    else return (static_cast<long>(p) * M1 + k) * N;
  };
  extern __shared__ float sm[];  // [M1][8 warps][4]
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long i0 = static_cast<long>(blockIdx.x) * kChunk + threadIdx.x * kElemsPerThread;
  const float* gp;
  if constexpr (kPerProblem) gp = g + vb;
  else gp = g + p * N;
  float gv[8], yv[8];
  load8(gp, i0, N, gv);
  const bool have_prev = st.n_iter >= 1;
  const int cand = st.cand_slot;
  if (have_prev) {
    float pv[8];
    if constexpr (kPerProblem) load8(g_prev + vb, i0, N, pv);
    else load8(g_prev + p * N, i0, N, pv);
#pragma unroll
    for (int j = 0; j < 8; ++j) yv[j] = hround(gv[j] - pv[j], Y);  // lbfgs.py:404
    hstore8(Y + hist(cand), i0, N, yv);
  } else {
#pragma unroll
    for (int j = 0; j < 8; ++j) yv[j] = 0.f;
  }
  // extras
  float gg = 0.f, g1 = 0.f, gm = 0.f;
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    gg = fmaf(gv[j], gv[j], gg);
    g1 += fabsf(gv[j]);
    gm = fmaxf(gm, fabsf(gv[j]));
  }
  gg = warp_sum(gg); g1 = warp_sum(g1); gm = warp_max(gm);
  __shared__ float sext[8][3];
  if (lane == 0) { sext[warp][0] = gg; sext[warp][1] = g1; sext[warp][2] = gm; }

  const int nlive = have_prev ? st.hist_count + 1 : 0;  // live pairs + candidate
  for (int k = 0; k < nlive; ++k) {
    const int slot = k < st.hist_count ? (st.hist_head + k) % M1 : cand;
    float sv[8], hv[8];
    hload8(S + hist(slot), i0, N, sv);
    if (slot == cand) {
#pragma unroll
      for (int j = 0; j < 8; ++j) hv[j] = yv[j];
    } else {
      hload8(Y + hist(slot), i0, N, hv);
    }
    float d0 = 0.f, d1 = 0.f, d2 = 0.f, d3 = 0.f;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      d0 = fmaf(sv[j], gv[j], d0);  // s_i . g
      d1 = fmaf(hv[j], gv[j], d1);  // y_i . g
      d2 = fmaf(sv[j], yv[j], d2);  // s_i . y_new
      d3 = fmaf(hv[j], yv[j], d3);  // y_i . y_new
    }
    d0 = warp_sum(d0); d1 = warp_sum(d1); d2 = warp_sum(d2); d3 = warp_sum(d3);
    if (lane == 0) {
      float* o = sm + (static_cast<long>(slot) * 8 + warp) * 4;
      o[0] = d0; o[1] = d1; o[2] = d2; o[3] = d3;
    }
  }
  __syncthreads();
  for (int t = threadIdx.x; t < nlive * 4; t += blockDim.x) {
    const int k = t >> 2, c = t & 3;
    const int slot = k < st.hist_count ? (st.hist_head + k) % M1 : cand;
    float acc = 0.f;
#pragma unroll
    for (int w = 0; w < 8; ++w) acc += sm[(static_cast<long>(slot) * 8 + w) * 4 + c];
    part[((static_cast<long>(p) * nblk + blockIdx.x) * M1 + slot) * 4 + c] = acc;
  }
  if (threadIdx.x < 3) {
    float acc = threadIdx.x == 2 ? 0.f : 0.f;
    for (int w = 0; w < 8; ++w) acc = threadIdx.x == 2 ? fmaxf(acc, sext[w][2]) : acc + sext[w][threadIdx.x];
    ext[(static_cast<long>(p) * nblk + blockIdx.x) * 4 + threadIdx.x] = acc;
  }
}

// ---------------------------------------------------------------------------------------------
// reduce the per-block partials: one block per (slot | extras, problem) -> dots[p][slot][4], dots[p][M1][0..2]
// (kept out of the control kernel: with 375+ partial blocks per image the serial sum was its latency floor)
// kPerProblem: problem p sums its own lbfgs_nblk(pr.vec_size(p)) partials; the rows stay nblk apart
// ---------------------------------------------------------------------------------------------
template <bool kPerProblem>
__global__ void __launch_bounds__(128)
lbfgs_reduce_kernel(const LbfgsState* __restrict__ states, const float* __restrict__ part,
                    const float* __restrict__ ext, int M1, int nblk, double* __restrict__ dots,
                    const __grid_constant__ ProblemArg<kPerProblem, ProblemRanges> pr) {
  const int p = blockIdx.y;
  const LbfgsState& st = states[p];
  if (st.done) return;
  int nb = nblk;   // partials of this problem
  if constexpr (kPerProblem) nb = nblk_of(pr.vec_size(p));
  const int slot = blockIdx.x;
  __shared__ double red[4][4];
  double a0 = 0, a1 = 0, a2 = 0, a3 = 0;
  if (slot < M1) {
    if (st.n_iter < 1) return;
    // live ring slots and the candidate only
    const int rel = (slot - st.hist_head + M1) % M1;
    if (!(rel < st.hist_count || slot == st.cand_slot)) return;
    for (int b = threadIdx.x; b < nb; b += blockDim.x) {
      const float4 q = __ldg(reinterpret_cast<const float4*>(part + ((static_cast<long>(p) * nblk + b) * M1 + slot) * 4));
      a0 += q.x; a1 += q.y; a2 += q.z; a3 += q.w;
    }
  } else {
    for (int b = threadIdx.x; b < nb; b += blockDim.x) {
      const float4 q = __ldg(reinterpret_cast<const float4*>(ext + (static_cast<long>(p) * nblk + b) * 4));
      a0 += q.x; a1 += q.y; a2 = fmax(a2, static_cast<double>(q.z));
    }
  }
  a0 = warp_sum(a0); a1 = warp_sum(a1); a3 = warp_sum(a3);
  if (slot < M1) a2 = warp_sum(a2);
  else
    for (int o = 16; o > 0; o >>= 1) a2 = fmax(a2, __shfl_xor_sync(0xffffffffu, a2, o));
  if ((threadIdx.x & 31) == 0) {
    red[threadIdx.x >> 5][0] = a0; red[threadIdx.x >> 5][1] = a1; red[threadIdx.x >> 5][2] = a2; red[threadIdx.x >> 5][3] = a3;
  }
  __syncthreads();
  if (threadIdx.x < 4) {
    const int c = threadIdx.x;
    double v;
    if (slot == M1 && c == 2) v = fmax(fmax(red[0][2], red[1][2]), fmax(red[2][2], red[3][2]));
    else v = red[0][c] + red[1][c] + red[2][c] + red[3][c];
    dots[(static_cast<long>(p) * (M1 + 1) + slot) * 4 + c] = v;
  }
}

// ---------------------------------------------------------------------------------------------
// control: one block (4 warps) per problem
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ double block_sum_128(double v, double* red) {
  v = warp_sum(v);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  return red[0] + red[1] + red[2] + red[3];
}

// kPerProblem: the loss weights of problem p are c_w[p], s_w[p] (device arrays) instead of cfg.c_weight, cfg.s_weight, and
// its losses are those of the images [pr.begin(p), pr.begin(p) + pr.size(p))
template <bool kPerProblem>
__global__ void __launch_bounds__(128)
lbfgs_control_kernel(LbfgsState* __restrict__ states, double* __restrict__ mats, const double* __restrict__ dots,
                     const double* __restrict__ loss_c,
                     const double* __restrict__ loss_s, int images_per_problem, int M1, LbfgsConfig cfg,
                     double* __restrict__ hist_c, double* __restrict__ hist_s, int tick, int P,
                     const double* __restrict__ c_w, const double* __restrict__ s_w,
                     const __grid_constant__ ProblemArg<kPerProblem, ProblemRanges> pr) {
  const int p = blockIdx.x;
  LbfgsState& st = states[p];
  __shared__ double red[4];
  __shared__ double sg[kMaxSlots], yg[kMaxSlots], syn[kMaxSlots], yyn[kMaxSlots];
  __shared__ double al[kMaxSlots], cs[kMaxSlots], cy[kMaxSlots];
  __shared__ int s_iter, s_commit;
  __shared__ double s_gamma;
  const int tid = threadIdx.x;

  // ---- losses of this evaluation (logged like pipelines.py:94-95) ----
  double lc = 0.0, ls = 0.0;
  if constexpr (kPerProblem) {
    const int first = pr.begin(p), g = pr.size(p);
    for (int i = tid; i < g; i += blockDim.x) {
      lc += loss_c[first + i];
      ls += loss_s[first + i];
    }
  } else {
    for (int i = tid; i < images_per_problem; i += blockDim.x) {
      lc += loss_c[p * images_per_problem + i];
      ls += loss_s[p * images_per_problem + i];
    }
  }
  lc = block_sum_128(lc, red);
  ls = block_sum_128(ls, red);
  (void)tick;  // the log row is the problem's own evaluation counter, so a captured CUDA graph can be replayed
  if (st.done) {
    if (tid == 0) { st.compute_d = 0; st.apply = 0; }
    return;
  }
  // ---- reduce the pass-1 partials ----
  const int M = cfg.history;
  const bool have_prev = st.n_iter >= 1;
  const int nlive = have_prev ? st.hist_count + 1 : 0;
  const double* dp = dots + static_cast<long>(p) * (M1 + 1) * 4;
  for (int k = tid; k < nlive; k += blockDim.x) {
    const int slot = k < st.hist_count ? (st.hist_head + k) % M1 : st.cand_slot;
    sg[slot] = dp[slot * 4 + 0]; yg[slot] = dp[slot * 4 + 1]; syn[slot] = dp[slot * 4 + 2]; yyn[slot] = dp[slot * 4 + 3];
  }
  const double gg = dp[M1 * 4 + 0], g1 = dp[M1 * 4 + 1], gm = dp[M1 * 4 + 2];
  __syncthreads();

  double* SY = mats + static_cast<long>(p) * 3 * M1 * M1;  // SY[i][j] = s_i . y_j
  double* SYT = SY + static_cast<long>(M1) * M1;           // SYT[j][i] = s_i . y_j
  double* YY = SYT + static_cast<long>(M1) * M1;

  // ---- state machine (lbfgs.py:364-374, 388-392, 504-526) ----
  if (tid == 0) {
    const double cw = kPerProblem ? c_w[p] : cfg.c_weight, sw = kPerProblem ? s_w[p] : cfg.s_weight;
    const double loss = cw * lc + sw * ls;
    st.last_c = lc; st.last_s = ls;
    hist_c[static_cast<long>(st.func_evals) * P + p] = lc;
    hist_s[static_cast<long>(st.func_evals) * P + p] = ls;
    st.func_evals += 1;
    st.loss = loss;
    int iterate = 0, end_step = 0;
    const bool opt_cond = gm <= cfg.tolerance_grad;
    if (st.phase == 0) {  // first closure of an optimizer.step
      st.current_evals = 1;
      if (opt_cond) end_step = 1;
      else { st.n_iter_step = 0; iterate = 1; }
    } else {              // re-evaluation after the update of iteration n_iter_step (< max_iter)
      st.current_evals += 1;
      const double max_td = static_cast<double>(__uint_as_float(st.max_td_bits));
      if (st.current_evals >= cfg.max_eval) end_step = 1;
      else if (opt_cond) end_step = 1;
      else if (max_td <= cfg.tolerance_change) end_step = 1;
      else if (fabs(loss - st.prev_loss) < cfg.tolerance_change) end_step = 1;
      else iterate = 1;
    }
    st.compute_d = 0; st.apply = 0;
    if (end_step) {
      st.phase = 0;
      if (st.func_evals >= cfg.epochs) st.done = 1;  // pipelines.py:79 re-checked between optim.step calls
    }
    s_iter = iterate;
    s_commit = 0;
    if (iterate) {
      st.n_iter_step += 1;
      st.n_iter += 1;
      if (st.n_iter == 1) {  // lbfgs.py:396-401
        st.hist_count = 0; st.hist_head = 0; st.cand_slot = 0; st.H_diag = 1.0;
      } else {
        const int c = st.cand_slot;
        const double ys = syn[c], yy = yyn[c];
        if (ys > 1e-10) {  // lbfgs.py:407-421
          if (st.hist_count == M) { st.hist_head = (st.hist_head + 1) % M1; st.hist_count -= 1; }
          st.hist_count += 1;
          st.ro[c] = 1.0 / ys;
          st.H_diag = ys / yy;
          s_commit = 1;
        }
      }
      s_gamma = st.H_diag;
    }
  }
  __syncthreads();
  if (!s_iter) return;
  const int cand_old = st.cand_slot;
  if (s_commit) {
    // new column of SY / new row+column of YY for the accepted pair (all live slots incl. itself)
    for (int k = tid; k < st.hist_count; k += blockDim.x) {
      const int slot = (st.hist_head + k) % M1;
      SY[static_cast<long>(slot) * M1 + cand_old] = syn[slot];
      SYT[static_cast<long>(cand_old) * M1 + slot] = syn[slot];
      YY[static_cast<long>(slot) * M1 + cand_old] = yyn[slot];
      YY[static_cast<long>(cand_old) * M1 + slot] = yyn[slot];
    }
    __syncthreads();
    if (tid == 0) st.cand_slot = (st.hist_head + st.hist_count) % M1;  // the free slot of the ring
  }
  __threadfence_block();
  __syncthreads();
  const int m = st.hist_count, head = st.hist_head;
  const double gamma = s_gamma;
  // ---- two-loop recursion in coefficient space (lbfgs.py:432-442), warp 0 ----
  // 2 m dependent steps, each a dot product of <= 100 terms against one matrix row in global memory (fp64).  The rows do
  // not depend on the recursion, so row k+1 is fetched into registers while row k is reduced, and the ring slots / ro
  // values are staged in shared memory once: measured with ncu at m = 100, 454 us -> 125 us per tick (on the critical path of
  // every problem: 1 % of a 640x400 tick, 5 % of a 224x224 one).  Same terms, same order, same results as the plain loops.
  // (An AXPY formulation -- lanes own rows, one broadcast per step, no reduction -- measured 142 us: not kept.)
  __shared__ int ring_slot[kMaxSlots];
  __shared__ double ro_s[kMaxSlots];
  for (int k = tid; k < m; k += blockDim.x) {
    const int sl = (head + k) % M1;
    ring_slot[k] = sl;
    ro_s[sl] = st.ro[sl];
  }
  __syncthreads();
  if (tid < 32) {
    // first loop: newest -> oldest; lane handles ring positions kk = k + 1 + tid + 32 t
    double rowv[4];
    auto fetch1 = [&](int k) {
      const long base = static_cast<long>(ring_slot[k]) * M1;
#pragma unroll
      for (int t = 0; t < 4; ++t) {
        const int kk = k + 1 + tid + 32 * t;
        rowv[t] = kk < m ? SY[base + ring_slot[kk]] : 0.0;
      }
    };
    if (m > 0) fetch1(m - 1);
    for (int k = m - 1; k >= 0; --k) {
      const int si = ring_slot[k];
      double cur[4];
#pragma unroll
      for (int t = 0; t < 4; ++t) cur[t] = rowv[t];
      if (k > 0) fetch1(k - 1);
      double acc = 0.0;
#pragma unroll
      for (int t = 0; t < 4; ++t) {
        const int kk = k + 1 + tid + 32 * t;
        if (kk < m) acc += al[ring_slot[kk]] * cur[t];
      }
      acc = warp_sum(acc);
      if (tid == 0) al[si] = ro_s[si] * (-sg[si] - acc);
      __syncwarp();
    }
    // second loop: oldest -> newest;  r = -gamma g - gamma sum al_j y_j + sum c_j s_j; lane handles kk = tid + 32 t
    double yyv[4], stv[4];
    auto fetch2 = [&](int k) {
      const long base = static_cast<long>(ring_slot[k]) * M1;
#pragma unroll
      for (int t = 0; t < 4; ++t) {
        const int kk = tid + 32 * t;
        yyv[t] = kk < m ? YY[base + ring_slot[kk]] : 0.0;
        stv[t] = kk < k ? SYT[base + ring_slot[kk]] : 0.0;
      }
    };
    if (m > 0) fetch2(0);
    for (int k = 0; k < m; ++k) {
      const int si = ring_slot[k];
      double cy_[4], cs_[4];
#pragma unroll
      for (int t = 0; t < 4; ++t) { cy_[t] = yyv[t]; cs_[t] = stv[t]; }
      if (k + 1 < m) fetch2(k + 1);
      double acc = 0.0;
#pragma unroll
      for (int t = 0; t < 4; ++t) {
        const int kk = tid + 32 * t;
        if (kk < m) {
          const int sj = ring_slot[kk];
          acc -= gamma * al[sj] * cy_[t];
          if (kk < k) acc += cs[sj] * cs_[t];  // y_i . s_j
        }
      }
      acc = warp_sum(acc);
      if (tid == 0) {
        const double be = ro_s[si] * (-gamma * yg[si] + acc);
        cs[si] = al[si] - be;
        cy[si] = -gamma * al[si];
      }
      __syncwarp();
    }
    // g . d  (lbfgs.py:460)
    double gtd = 0.0;
    for (int kk = tid; kk < m; kk += 32) {
      const int sj = (head + kk) % M1;
      gtd += cs[sj] * sg[sj] + cy[sj] * yg[sj];
    }
    gtd = warp_sum(gtd);
    for (int kk = tid; kk < m; kk += 32) {
      const int sj = (head + kk) % M1;
      st.coef_s[sj] = static_cast<float>(cs[sj]);
      st.coef_y[sj] = static_cast<float>(cy[sj]);
    }
    if (tid == 0) {
      gtd += -gamma * gg;
      st.coef_g = static_cast<float>(-gamma);
      st.prev_loss = st.loss;  // lbfgs.py:448
      const double t = st.n_iter == 1 ? fmin(1.0, 1.0 / g1) * cfg.lr : cfg.lr;  // lbfgs.py:454-457
      st.t = t;
      st.compute_d = 1;
      st.max_td_bits = 0u;
      if (gtd > -cfg.tolerance_change) {  // lbfgs.py:463: break before the update
        st.apply = 0;
        st.phase = 0;
        if (st.func_evals >= cfg.epochs) st.done = 1;
      } else {
        st.apply = 1;
        if (st.n_iter_step != cfg.max_iter) st.phase = 1;
        else {
          st.phase = 0;
          if (st.func_evals >= cfg.epochs) st.done = 1;
        }
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------
// pass 2
// ---------------------------------------------------------------------------------------------
// kPerProblem: the slices of lbfgs_dots_kernel
template <typename HT, bool kPerProblem>
__global__ void __launch_bounds__(kDotThreads)
lbfgs_update_kernel(float* __restrict__ x, const float* __restrict__ g, float* __restrict__ g_prev,
                    HT* __restrict__ S, const HT* __restrict__ Y, LbfgsState* __restrict__ states, long N,
                    int M1, const __grid_constant__ ProblemArg<kPerProblem, ProblemRanges> pr) {
  const int p = blockIdx.y;
  LbfgsState& st = states[p];
  if (!st.compute_d) return;
  long vb;
  if constexpr (kPerProblem) {
    vb = pr.vec_begin(p);
    N = pr.vec_size(p);
    if (static_cast<int>(blockIdx.x) >= nblk_of(N)) return;
  }
  auto hist = [&](int k) -> long {
    if constexpr (kPerProblem) return M1 * vb + k * N;
    else return (static_cast<long>(p) * M1 + k) * N;
  };
  auto vec = [&]() -> long {
    if constexpr (kPerProblem) return vb;
    else return p * N;
  };
  const long i0 = static_cast<long>(blockIdx.x) * kChunk + threadIdx.x * kElemsPerThread;
  float gv[8], d[8];
  load8(g + vec(), i0, N, gv);
  const float cg = st.coef_g;
#pragma unroll
  for (int j = 0; j < 8; ++j) d[j] = cg * gv[j];
  const int m = st.hist_count, head = st.hist_head;
  for (int k = 0; k < m; ++k) {
    const int slot = (head + k) % M1;
    const float a = st.coef_s[slot], b = st.coef_y[slot];
    float sv[8], yv[8];
    hload8(S + hist(slot), i0, N, sv);
    hload8(Y + hist(slot), i0, N, yv);
#pragma unroll
    for (int j = 0; j < 8; ++j) d[j] = fmaf(a, sv[j], fmaf(b, yv[j], d[j]));
  }
  const float t = static_cast<float>(st.t);
  float sv[8];
  float mx = 0.f;
#pragma unroll
  for (int j = 0; j < 8; ++j) { sv[j] = d[j] * t; mx = fmaxf(mx, fabsf(sv[j])); }  // s = d.mul(t), lbfgs.py:405
  hstore8(S + hist(st.cand_slot), i0, N, sv);
  store8(g_prev + vec(), i0, N, gv);  // lbfgs.py:444-447
  if (st.apply) {
    float xv[8];
    load8(x + vec(), i0, N, xv);
#pragma unroll
    for (int j = 0; j < 8; ++j) xv[j] = fminf(fmaxf(fmaf(t, d[j], xv[j]), 0.f), 1.f);  // lbfgs.py:313 + pipelines.py:82
    store8(x + vec(), i0, N, xv);
  }
  mx = warp_max(mx);
  if ((threadIdx.x & 31) == 0 && mx > 0.f) atomicMax(&st.max_td_bits, __float_as_uint(mx));
}

__global__ void clamp01_kernel(float* __restrict__ x, long n) {
  for (long i = blockIdx.x * static_cast<long>(blockDim.x) + threadIdx.x; i < n;
       i += static_cast<long>(gridDim.x) * blockDim.x)
    x[i] = fminf(fmaxf(x[i], 0.f), 1.f);
}

__global__ void lbfgs_init_kernel(LbfgsState* states, int P) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= P) return;
  LbfgsState& st = states[p];
  st.n_iter = 0; st.func_evals = 0; st.phase = 0; st.n_iter_step = 0; st.current_evals = 0;
  st.hist_count = 0; st.hist_head = 0; st.cand_slot = 0; st.done = 0; st.compute_d = 0; st.apply = 0;
  st.max_td_bits = 0u; st.loss = 0; st.prev_loss = 0; st.t = 0; st.H_diag = 1.0; st.last_c = 0; st.last_s = 0;
  st.coef_g = 0.f;
}

int lbfgs_nblk(long N) { return nblk_of(N); }

int lbfgs_init(LbfgsState* states, int P, cudaStream_t s) {
  lbfgs_init_kernel<<<(P + 127) / 128, 128, 0, s>>>(states, P);
  ISX_LAUNCH_CHECK();
  return 0;
}

int clamp01(float* x, long n, cudaStream_t s) {
  const int blocks = static_cast<int>(std::min<long>((n + 255) / 256, static_cast<long>(isx_num_sms()) * 8));
  clamp01_kernel<<<blocks, 256, 0, s>>>(x, n);
  ISX_LAUNCH_CHECK();
  return 0;
}

int lbfgs_tick(float* x, const float* g, float* g_prev, void* S, void* Y, int history_bf16, LbfgsState* states, double* mats,
               float* part, float* ext, double* dots, const double* loss_c, const double* loss_s, int images_per_problem, int P,
               long N, const LbfgsConfig& cfg, double* hist_c, double* hist_s, int tick, cudaStream_t s, const double* c_w,
               const double* s_w, const ProblemRanges* pr) {
  const int M1 = cfg.history + 1;
  ISX_REQUIRE(M1 <= kMaxSlots, "lbfgs: history %d exceeds %d", cfg.history, kMaxSlots - 1);
  const int nblk = lbfgs_nblk(N);
  dim3 grid(nblk, P);
  const size_t sm1 = static_cast<size_t>(M1) * 8 * 4 * sizeof(float);
  isx_prof_begin(ISX_PROF_LBFGS, 0.0, s);  // both history passes + control; bytes are derived by the caller
  if (pr) {   // several problems with their own weights: grid over the largest problem (N), slices from the descriptor
    if (history_bf16)
      lbfgs_dots_kernel<__nv_bfloat16, true><<<grid, kDotThreads, sm1, s>>>(
          g, g_prev, static_cast<const __nv_bfloat16*>(S), static_cast<__nv_bfloat16*>(Y), states, N, M1, nblk, part, ext, *pr);
    else
      lbfgs_dots_kernel<float, true><<<grid, kDotThreads, sm1, s>>>(g, g_prev, static_cast<const float*>(S),
                                                                    static_cast<float*>(Y), states, N, M1, nblk, part, ext, *pr);
    ISX_LAUNCH_CHECK();
    lbfgs_reduce_kernel<true><<<dim3(M1 + 1, P), 128, 0, s>>>(states, part, ext, M1, nblk, dots, *pr);
    ISX_LAUNCH_CHECK();
    lbfgs_control_kernel<true><<<P, 128, 0, s>>>(states, mats, dots, loss_c, loss_s, images_per_problem, M1, cfg, hist_c,
                                                 hist_s, tick, P, c_w, s_w, *pr);
    ISX_LAUNCH_CHECK();
    if (history_bf16)
      lbfgs_update_kernel<__nv_bfloat16, true><<<grid, kDotThreads, 0, s>>>(
          x, g, g_prev, static_cast<__nv_bfloat16*>(S), static_cast<const __nv_bfloat16*>(Y), states, N, M1, *pr);
    else
      lbfgs_update_kernel<float, true><<<grid, kDotThreads, 0, s>>>(x, g, g_prev, static_cast<float*>(S),
                                                                    static_cast<const float*>(Y), states, N, M1, *pr);
  } else {
    if (history_bf16)
      lbfgs_dots_kernel<__nv_bfloat16, false><<<grid, kDotThreads, sm1, s>>>(
          g, g_prev, static_cast<const __nv_bfloat16*>(S), static_cast<__nv_bfloat16*>(Y), states, N, M1, nblk, part, ext,
          NoProblems());
    else
      lbfgs_dots_kernel<float, false><<<grid, kDotThreads, sm1, s>>>(g, g_prev, static_cast<const float*>(S),
                                                                     static_cast<float*>(Y), states, N, M1, nblk, part, ext,
                                                                     NoProblems());
    ISX_LAUNCH_CHECK();
    lbfgs_reduce_kernel<false><<<dim3(M1 + 1, P), 128, 0, s>>>(states, part, ext, M1, nblk, dots, NoProblems());
    ISX_LAUNCH_CHECK();
    lbfgs_control_kernel<false><<<P, 128, 0, s>>>(states, mats, dots, loss_c, loss_s, images_per_problem, M1, cfg, hist_c,
                                                  hist_s, tick, P, nullptr, nullptr, NoProblems());
    ISX_LAUNCH_CHECK();
    if (history_bf16)
      lbfgs_update_kernel<__nv_bfloat16, false><<<grid, kDotThreads, 0, s>>>(
          x, g, g_prev, static_cast<__nv_bfloat16*>(S), static_cast<const __nv_bfloat16*>(Y), states, N, M1, NoProblems());
    else
      lbfgs_update_kernel<float, false><<<grid, kDotThreads, 0, s>>>(x, g, g_prev, static_cast<float*>(S),
                                                                     static_cast<const float*>(Y), states, N, M1, NoProblems());
  }
  isx_prof_end(ISX_PROF_LBFGS, s);
  ISX_LAUNCH_CHECK();
  return 0;
}

}  // namespace isx
