// Internal launchers of the HBM-bound kernels (elementwise.cu, lbfgs.cu, imageops.cu).
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <type_traits>

namespace isx {

int pack_conv_weights(const float* w, int Cout, int Cin, __nv_bfloat16* wf, __nv_bfloat16* wd, cudaStream_t s);
int pack_w0_dgrad(const float* w, __nv_bfloat16* wd, cudaStream_t s);
int pack_w0_fwd(const float* w, __nv_bfloat16* wp, cudaStream_t s);
int conv1_1_fwd_tc(const float* x, int xc, const float* mask, int mask_b, const __nv_bfloat16* w0_packed,
                   const float* bias, __nv_bfloat16* out, int B, int H, int W, cudaStream_t s);
int conv1_1_fwd(const float* x, int xc, const float* mask, int mask_b, const float* w, const float* bias,
                __nv_bfloat16* out, int B, int H, int W, cudaStream_t s);
int conv1_1_dgrad(const __nv_bfloat16* dy, const float* w, const float* mask, int mask_b, float* dx, int xc, int B,
                  int H, int W, cudaStream_t s);
int maxpool_fwd(const __nv_bfloat16* in, __nv_bfloat16* out, int B, int H, int W, int C, cudaStream_t s);
int maxpool_bwd(const __nv_bfloat16* dy, const __nv_bfloat16* act, __nv_bfloat16* dx, int B, int H, int W, int C,
                cudaStream_t s);
// the pool with the routing codes of its backward (one byte per pooled element: 0..3 first maximum, 4 blocked by the ReLU)
int maxpool_fwd_idx(const __nv_bfloat16* in, __nv_bfloat16* out, uint8_t* idx, int B, int H, int W, int C, cudaStream_t s);
int maxpool_bwd_idx(const __nv_bfloat16* dy, const uint8_t* idx, __nv_bfloat16* dx, int B, int H, int W, int C,
                    cudaStream_t s);
int tap_add_mask(const __nv_bfloat16* g, const __nv_bfloat16* add, const float* aff_a, const float* aff_b,
                 const __nv_bfloat16* act, __nv_bfloat16* out, int B, long HW, int C, cudaStream_t s, int relu_mask = 1);
int mask_features(const __nv_bfloat16* f, const float* m, int mask_b, __nv_bfloat16* fm, __nv_bfloat16* fm2, int B,
                  long HW, int C, cudaStream_t s);
int avgpool2x2_f32(const float* in, float* out, int B, int H, int W, cudaStream_t s);
// Several coupled problems in one batch: problem p is the images [begin(p), begin(p + 1)).  Equal problems
// (isx_nst_eval_problems, isx_lbfgs_tick_problems) derive the ranges from ipp; problems of unequal size
// (isx_nst_eval_ranges, isx_lbfgs_tick_ranges) carry the validated host offsets by value, so a captured launch needs no
// device allocation.  Kernels take the descriptor as a __grid_constant__ parameter and index it in the constant bank.
static constexpr int kMaxRangedProblems = 1024;  // == ISX_MAX_RANGED_PROBLEMS
struct ProblemRanges {
  int P = 0;
  int ipp = 0;     // > 0: problem p is the images [p * ipp, (p + 1) * ipp) and first[] is not read
  long n = 0;      // L-BFGS passes: floats of one problem (ipp > 0) or of one image (ipp == 0)
  int first[kMaxRangedProblems + 1];
  __host__ __device__ __forceinline__ int begin(int p) const { return ipp ? p * ipp : first[p]; }
  __host__ __device__ __forceinline__ int size(int p) const { return ipp ? ipp : first[p + 1] - first[p]; }
  __device__ __forceinline__ int problem_of(int b) const {
    if (ipp) return b / ipp;
    int lo = 0, hi = P - 1;          // the last p with first[p] <= b
    while (lo < hi) {
      const int mid = (lo + hi + 1) >> 1;
      if (first[mid] <= b) lo = mid;
      else hi = mid - 1;
    }
    return lo;
  }
  // the slice of the parameter vector (x, g, g_prev) that problem p owns, in floats; its S / Y block starts at M1 * vec_begin
  __device__ __forceinline__ long vec_begin(int p) const { return ipp ? p * n : first[p] * n; }
  __device__ __forceinline__ long vec_size(int p) const { return ipp ? n : (first[p + 1] - first[p]) * n; }
};
// Each finalize kernel forms image b's gradient scale from weight[p(b)], k1 and k2 with the same double operations the host
// uses for its scalar grad_scale, so that one problem's images match a scalar call bit for bit.
struct ProblemWeights {
  const double* weight = nullptr;  // device [P]: alpha (content) or beta (style) per problem
  int target = 0;                  // style target of image b: 0 the shared one, 1 its problem's, 2 its own
  double k1 = 0.0, k2 = 0.0;
  ProblemRanges r;
  __device__ __forceinline__ int target_of(int b, int p) const { return target == 0 ? 0 : target == 1 ? p : b; }
};
// what the scalar instantiations (kPerProblem = false) take in place of a descriptor
struct NoProblems {};
template <bool kPerProblem, class T>
using ProblemArg = typename std::conditional<kPerProblem, T, NoProblems>::type;
int gram_finalize(const float* partial, int B, int splits, int C, float inv_n, float* G_out, const float* target,
                  int target_b, double loss_scale, double* loss, float grad_scale, __nv_bfloat16* D_out,
                  cudaStream_t s, float* triu = nullptr, long triu_ld = 0, const ProblemWeights* pw = nullptr);
int content_mse(const __nv_bfloat16* pred, const __nv_bfloat16* target, int target_b, __nv_bfloat16* grad, int B,
                long per_image, double loss_scale, float grad_scale, double* loss, cudaStream_t s, int relu_mask = 1,
                const ProblemWeights* pw = nullptr);
int chan_sums(const __nv_bfloat16* f, int B, long HW, int C, double* sums, cudaStream_t s, const float* mask = nullptr,
              int mask_b = 0);
int masked_affine_grad(const __nv_bfloat16* f, const float* m, int mask_b, const float* aff_a, const float* aff_b,
                       __nv_bfloat16* out, int B, long HW, int C, cudaStream_t s);
int stats_from_gram(const float* partial, const float* csum, int B, int splits, int C, long HW, float* mean, float* stdv,
                    long out_ld, cudaStream_t s);
int bn_finalize(const double* sums, int B, int C, long HW, float* mean, float* stdv, const float* t_mean,
                const float* t_std, int target_b, double loss_scale, double grad_scale, double* loss, float* aff_a,
                float* aff_b, cudaStream_t s, long out_ld = 0,   // out_ld: row stride of mean / stdv (0 = C)
                const ProblemWeights* pw = nullptr);

}  // namespace isx
