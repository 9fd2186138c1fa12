// Internal launchers of the HBM-bound kernels (elementwise.cu, lbfgs.cu, imageops.cu).
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

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
// Several coupled problems in one batch (isx_nst_eval_problems): image b belongs to problem b / ipp and scales its loss
// gradient by that problem's weight.  Each finalize kernel forms the scale from weight[p], k1 and k2 with the same double
// operations the host uses for its scalar grad_scale, so that one problem's images match a scalar call bit for bit.
struct ProblemWeights {
  const double* weight = nullptr;  // device [P]: alpha (content) or beta (style) per problem
  int ipp = 1;                     // images per problem
  int target_div = 1;              // image b reads style target b / target_div (B / style target batch)
  double k1 = 0.0, k2 = 0.0;
};
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
