// C-ABI wrappers (include/isx.h) over the kernel launchers.
#include "../../include/isx.h"
#include "isx_common.cuh"
#include "isx_internal.h"
#include "isx_kernels.h"

using namespace isx;
typedef __nv_bfloat16 bf16;

static inline cudaStream_t S(isx_stream s) { return reinterpret_cast<cudaStream_t>(s); }
static inline const bf16* P(const isx_bf16* p) { return reinterpret_cast<const bf16*>(p); }
static inline bf16* P(isx_bf16* p) { return reinterpret_cast<bf16*>(p); }

// tile_cfg (test / tuning hook): BN*100 + MT*10 + stages forces that tile of the generic kernel (conv_tc.cu);
// 0 = library heuristic (conv_c64 / conv_halo / generic).  E.g. 25623 = BN 256, MT 2, 3 stages.
static void decode_tile_cfg(int cfg, ConvArgs* a) {
  if (cfg > 0) {
    a->force_bn = cfg / 100;
    a->force_mt = (cfg % 100) / 10;
    a->force_stages = cfg % 10;
  }
}

extern "C" int isx_pack_conv3x3_weights(const float* w, int Cout, int Cin, isx_bf16* wf, isx_bf16* wd,
                                        isx_stream stream) {
  ISX_REQUIRE(w && (wf || wd) && Cout > 0 && Cin > 0, "isx_pack_conv3x3_weights: bad arguments");
  return pack_conv_weights(w, Cout, Cin, P(wf), P(wd), S(stream));
}

extern "C" int isx_conv1_1_fwd(const float* x, int xc, const float* mask, int mask_b, const float* w,
                               const float* bias, isx_bf16* out, int B, int H, int W, isx_stream stream) {
  ISX_REQUIRE(x && w && out && B > 0 && H > 0 && W > 0, "isx_conv1_1_fwd: bad arguments");
  ISX_REQUIRE(!mask || mask_b == 1 || mask_b == B, "isx_conv1_1_fwd: mask batch %d must be 1 or %d", mask_b, B);
  return conv1_1_fwd(x, xc, mask, mask_b, w, bias, P(out), B, H, W, S(stream));
}

extern "C" int isx_pack_conv1_1_fwd(const float* w, isx_bf16* w0_fwd, isx_stream stream) {
  ISX_REQUIRE(w && w0_fwd, "isx_pack_conv1_1_fwd: null pointer");
  return pack_w0_fwd(w, P(w0_fwd), S(stream));
}

extern "C" int isx_conv1_1_fwd_tc(const float* x, int xc, const float* mask, int mask_b, const isx_bf16* w0_fwd,
                                  const float* bias, isx_bf16* out, int B, int H, int W, isx_stream stream) {
  ISX_REQUIRE(x && w0_fwd && out && B > 0 && H > 0 && W > 0, "isx_conv1_1_fwd_tc: bad arguments");
  ISX_REQUIRE(!mask || mask_b == 1 || mask_b == B, "isx_conv1_1_fwd_tc: mask batch %d must be 1 or %d", mask_b, B);
  return conv1_1_fwd_tc(x, xc, mask, mask ? mask_b : 0, P(w0_fwd), bias, P(out), B, H, W, S(stream));
}

extern "C" int isx_pack_conv1_1_dgrad(const float* w, isx_bf16* w0_dgrad, isx_stream stream) {
  ISX_REQUIRE(w && w0_dgrad, "isx_pack_conv1_1_dgrad: null pointer");
  return pack_w0_dgrad(w, P(w0_dgrad), S(stream));
}

extern "C" int isx_conv1_1_dgrad_tc(const isx_bf16* dy, const isx_bf16* w0_dgrad, const float* mask, int mask_b,
                                    float* dx, int xc, int B, int H, int W, isx_stream stream) {
  ISX_REQUIRE(dy && w0_dgrad && dx && B > 0 && H > 0 && W > 0, "isx_conv1_1_dgrad_tc: bad arguments");
  ISX_REQUIRE(!mask || mask_b == 1 || mask_b == B, "isx_conv1_1_dgrad_tc: mask batch %d must be 1 or %d", mask_b, B);
  ConvArgs a;
  a.in = P(dy); a.weight = P(w0_dgrad); a.out = nullptr;
  a.B = B; a.H = H; a.W = W; a.Cin = 64; a.Cout = 16; a.ntaps = 9;
  a.dx_nchw = dx; a.xc = xc; a.in_mask = mask; a.mask_b = mask ? mask_b : 0;
  return conv_tc(a, S(stream));
}

extern "C" int isx_conv1_1_dgrad(const isx_bf16* dy, const float* w, const float* mask, int mask_b, float* dx, int xc,
                                 int B, int H, int W, isx_stream stream) {
  ISX_REQUIRE(dy && w && dx && B > 0 && H > 0 && W > 0, "isx_conv1_1_dgrad: bad arguments");
  ISX_REQUIRE(xc == 1 || xc == 3, "isx_conv1_1_dgrad: xc must be 1 or 3");
  return conv1_1_dgrad(P(dy), w, mask, mask_b, dx, xc, B, H, W, S(stream));
}

extern "C" int isx_conv3x3_bias_relu_fwd(const isx_bf16* in, const isx_bf16* w_fwd, const float* bias, isx_bf16* out,
                                         int B, int H, int W, int Cin, int Cout, int relu, int tile_cfg,
                                         isx_stream stream) {
  ISX_REQUIRE(in && w_fwd && out, "isx_conv3x3_bias_relu_fwd: null pointer");
  ConvArgs a;
  a.in = P(in); a.weight = P(w_fwd); a.out = P(out);
  a.B = B; a.H = H; a.W = W; a.Cin = Cin; a.Cout = Cout; a.ntaps = 9;
  a.bias = bias; a.relu = relu;
  decode_tile_cfg(tile_cfg, &a);
  return conv_tc(a, S(stream));
}

extern "C" int isx_conv3x3_bias_relu_pool_fwd(const isx_bf16* in, const isx_bf16* w_fwd, const float* bias, isx_bf16* out,
                                              isx_bf16* pool_out, int B, int H, int W, int Cin, int Cout, int tile_cfg,
                                              isx_stream stream) {
  ISX_REQUIRE(in && w_fwd && out && pool_out && H >= 2 && W >= 2, "isx_conv3x3_bias_relu_pool_fwd: bad arguments");
  ConvArgs a;
  a.in = P(in); a.weight = P(w_fwd); a.out = P(out); a.pool_out = P(pool_out);
  a.B = B; a.H = H; a.W = W; a.Cin = Cin; a.Cout = Cout; a.ntaps = 9;
  a.bias = bias; a.relu = 1;
  decode_tile_cfg(tile_cfg, &a);
  return conv_tc(a, S(stream));
}

extern "C" int isx_conv3x3_bias_relu_pool_idx_fwd(const isx_bf16* in, const isx_bf16* w_fwd, const float* bias, isx_bf16* out,
                                                  isx_bf16* pool_out, uint8_t* pool_idx, int skip_out, int B, int H, int W,
                                                  int Cin, int Cout, int tile_cfg, isx_stream stream) {
  ISX_REQUIRE(in && w_fwd && out && pool_out && pool_idx && H >= 2 && W >= 2, "isx_conv3x3_bias_relu_pool_idx_fwd: bad arguments");
  ConvArgs a;
  a.in = P(in); a.weight = P(w_fwd); a.out = P(out); a.pool_out = P(pool_out); a.pool_idx = pool_idx; a.skip_out = skip_out != 0;
  a.B = B; a.H = H; a.W = W; a.Cin = Cin; a.Cout = Cout; a.ntaps = 9;
  a.bias = bias; a.relu = 1;
  decode_tile_cfg(tile_cfg, &a);
  return conv_tc(a, S(stream));
}

extern "C" int isx_conv3x3_dgrad(const isx_bf16* dy, const isx_bf16* w_dgrad, isx_bf16* dx, int B, int H, int W,
                                 int Cin, int Cout, const isx_bf16* relu_act, const isx_bf16* add_grad,
                                 const float* aff_a, const float* aff_b, int tile_cfg, isx_stream stream) {
  ISX_REQUIRE(dy && w_dgrad && dx, "isx_conv3x3_dgrad: null pointer");
  ConvArgs a;
  a.in = P(dy); a.weight = P(w_dgrad); a.out = P(dx);
  a.B = B; a.H = H; a.W = W; a.Cin = Cout; a.Cout = Cin; a.ntaps = 9;  // GEMM K = fwd Cout, N = fwd Cin
  a.mask_act = P(relu_act); a.add_buf = P(add_grad); a.aff_a = aff_a; a.aff_b = aff_b;
  decode_tile_cfg(tile_cfg, &a);
  return conv_tc(a, S(stream));
}

extern "C" int isx_conv3x3_dgrad_gram(const isx_bf16* dy, const isx_bf16* w_dgrad, isx_bf16* dx, int B, int H, int W,
                                      int Cin, int Cout, const isx_bf16* act_below, const isx_bf16* gram_D,
                                      isx_stream stream) {
  ISX_REQUIRE(dy && w_dgrad && dx && act_below && gram_D, "isx_conv3x3_dgrad_gram: null pointer");
  ConvArgs a;
  a.in = P(dy); a.weight = P(w_dgrad); a.out = P(dx);
  a.B = B; a.H = H; a.W = W; a.Cin = Cout; a.Cout = Cin; a.ntaps = 9;
  a.mask_act = P(act_below); a.gram_act = P(act_below); a.gram_D = P(gram_D);
  return conv_tc(a, S(stream));
}

extern "C" int isx_maxpool2x2_fwd(const isx_bf16* in, isx_bf16* out, int B, int H, int W, int C, isx_stream stream) {
  ISX_REQUIRE(in && out, "isx_maxpool2x2_fwd: null pointer");
  return maxpool_fwd(P(in), P(out), B, H, W, C, S(stream));
}

extern "C" int isx_maxpool2x2_bwd(const isx_bf16* dy, const isx_bf16* act, isx_bf16* dx, int B, int H, int W, int C,
                                  isx_stream stream) {
  ISX_REQUIRE(dy && act && dx, "isx_maxpool2x2_bwd: null pointer");
  return maxpool_bwd(P(dy), P(act), P(dx), B, H, W, C, S(stream));
}

extern "C" int isx_maxpool2x2_fwd_idx(const isx_bf16* in, isx_bf16* out, uint8_t* idx, int B, int H, int W, int C,
                                      isx_stream stream) {
  ISX_REQUIRE(in && idx, "isx_maxpool2x2_fwd_idx: null pointer");
  return maxpool_fwd_idx(P(in), P(out), idx, B, H, W, C, S(stream));
}

extern "C" int isx_maxpool2x2_bwd_idx(const isx_bf16* dy, const uint8_t* idx, isx_bf16* dx, int B, int H, int W, int C,
                                      isx_stream stream) {
  ISX_REQUIRE(dy && idx && dx, "isx_maxpool2x2_bwd_idx: null pointer");
  return maxpool_bwd_idx(P(dy), idx, P(dx), B, H, W, C, S(stream));
}

extern "C" int64_t isx_gram_workspace_bytes(int B, int HW, int C) {
  if (B <= 0 || HW <= 0 || C <= 0) return 0;
  return static_cast<int64_t>(gram_pick_splits(B, HW, C)) * B * C * C * 4;
}

extern "C" int isx_gram_fwd(const isx_bf16* feat, int B, int HW, int C, float inv_n, void* workspace, float* G_out,
                            const float* target, int target_b, double loss_scale, double* loss, float grad_scale,
                            isx_bf16* D_out, isx_stream stream) {
  ISX_REQUIRE(feat && workspace, "isx_gram_fwd: null pointer");
  ISX_REQUIRE(!target || target_b == 1 || target_b == B, "isx_gram_fwd: target batch %d must be 1 or %d", target_b, B);
  const int splits = gram_pick_splits(B, HW, C);
  int rc = gram_tc_partial(P(feat), B, HW, C, splits, static_cast<float*>(workspace), S(stream));
  if (rc) return rc;
  return gram_finalize(static_cast<const float*>(workspace), B, splits, C, inv_n, G_out, target, target_b, loss_scale,
                       loss, grad_scale, P(D_out), S(stream));
}

extern "C" int64_t isx_gram_mask_flags_bytes(int mask_b, int HW, int C) {
  if (mask_b <= 0 || HW <= 0 || C <= 0) return 0;
  return gram_mask_flags_bytes(mask_b, HW, C);
}

extern "C" int isx_gram_masked_fwd(const isx_bf16* feat, int B, int HW, int C, const float* m, int mask_b, void* flags_ws,
                                   isx_bf16* fm2, float inv_n, void* workspace, float* G_out, const float* target,
                                   int target_b, double loss_scale, double* loss, float grad_scale, isx_bf16* D_out,
                                   isx_stream stream) {
  ISX_REQUIRE(feat && m && flags_ws && workspace, "isx_gram_masked_fwd: null pointer");
  ISX_REQUIRE(mask_b == 1 || mask_b == B, "isx_gram_masked_fwd: mask batch %d must be 1 or %d", mask_b, B);
  ISX_REQUIRE(!target || target_b == 1 || target_b == B, "isx_gram_masked_fwd: target batch %d must be 1 or %d", target_b, B);
  int rc = gram_mask_flags(m, mask_b, HW, C, static_cast<uint8_t*>(flags_ws), S(stream));
  if (rc) return rc;
  ISX_REQUIRE(fm2 != nullptr, "isx_gram_masked_fwd: fm2 (bf16 [B,HW,C]) is required: the kernel stores F*m^2 while it scales the tiles");
  ISX_CHECK_CUDA(cudaMemsetAsync(fm2, 0, static_cast<size_t>(B) * HW * C * 2, S(stream)));
  GramMask gm;
  gm.m = m; gm.mask_b = mask_b; gm.kb_flags = static_cast<const uint8_t*>(flags_ws); gm.fm2 = P(fm2);
  const int splits = gram_pick_splits(B, HW, C);
  rc = gram_sym_partial(P(feat), B, HW, C, splits, static_cast<float*>(workspace), &gm, S(stream));
  if (rc) return rc;
  return gram_finalize(static_cast<const float*>(workspace), B, splits, C, inv_n, G_out, target, target_b, loss_scale,
                       loss, grad_scale, P(D_out), S(stream));
}

extern "C" int isx_gram_bwd(const isx_bf16* feat, const isx_bf16* D, isx_bf16* dF, int B, int H, int W, int C,
                            const isx_bf16* relu_act, isx_stream stream) {
  ISX_REQUIRE(feat && D && dF, "isx_gram_bwd: null pointer");
  ConvArgs a;
  a.in = P(feat); a.weight = P(D); a.out = P(dF);
  a.B = B; a.H = H; a.W = W; a.Cin = C; a.Cout = C; a.ntaps = 1;
  a.per_image_weights = true;
  a.mask_act = P(relu_act);
  return conv_tc(a, S(stream));
}

extern "C" int isx_content_mse_fwd_bwd(const isx_bf16* pred, const isx_bf16* target, int target_b, isx_bf16* grad,
                                       int B, int64_t per_image, double loss_scale, float grad_scale, double* loss,
                                       isx_stream stream) {
  ISX_REQUIRE(pred && target && loss, "isx_content_mse_fwd_bwd: null pointer");
  ISX_REQUIRE(target_b == 1 || target_b == B, "isx_content_mse_fwd_bwd: target batch %d must be 1 or %d", target_b, B);
  return content_mse(P(pred), P(target), target_b, P(grad), B, per_image, loss_scale, grad_scale, loss, S(stream));
}

extern "C" int isx_mse_fwd_bwd(const isx_bf16* pred, const isx_bf16* target, int target_b, isx_bf16* grad, int B,
                               int64_t per_image, double loss_scale, float grad_scale, int relu_mask, double* loss,
                               isx_stream stream) {
  ISX_REQUIRE(pred && target && loss, "isx_mse_fwd_bwd: null pointer");
  ISX_REQUIRE(target_b == 1 || target_b == B, "isx_mse_fwd_bwd: target batch %d must be 1 or %d", target_b, B);
  return content_mse(P(pred), P(target), target_b, P(grad), B, per_image, loss_scale, grad_scale, loss, S(stream), relu_mask);
}

extern "C" int isx_channel_affine(const isx_bf16* feat, const float* a, const float* b, isx_bf16* out, int B, int64_t HW, int C,
                                  int relu_mask, isx_stream stream) {
  ISX_REQUIRE(feat && a && b && out && C % 8 == 0, "isx_channel_affine: bad arguments");
  return tap_add_mask(nullptr, nullptr, a, b, P(feat), P(out), B, HW, C, S(stream), relu_mask);
}

extern "C" int isx_bn_stats_fwd(const isx_bf16* feat, int B, int64_t HW, int C, double* sums, float* mean, float* std_,
                                const float* t_mean, const float* t_std, int target_b, double loss_scale,
                                double grad_scale, double* loss, float* aff_a, float* aff_b, isx_stream stream) {
  ISX_REQUIRE(feat && sums, "isx_bn_stats_fwd: null pointer");
  ISX_REQUIRE(HW >= 2, "isx_bn_stats_fwd: unbiased std needs at least 2 pixels");
  ISX_CHECK_CUDA(cudaMemsetAsync(sums, 0, static_cast<size_t>(B) * C * 2 * sizeof(double), S(stream)));
  int rc = chan_sums(P(feat), B, HW, C, sums, S(stream));
  if (rc) return rc;
  return bn_finalize(sums, B, C, HW, mean, std_, t_mean, t_std, target_b, loss_scale, grad_scale, loss, aff_a, aff_b,
                     S(stream));
}

extern "C" int isx_bn_stats_masked_fwd(const isx_bf16* feat, const float* m, int mask_b, int B, int64_t HW, int C, double* sums,
                                       float* mean, float* std_, isx_stream stream) {
  ISX_REQUIRE(feat && m && sums && mean && std_, "isx_bn_stats_masked_fwd: null pointer");
  ISX_REQUIRE(mask_b == 1 || mask_b == B, "isx_bn_stats_masked_fwd: mask batch %d must be 1 or %d", mask_b, B);
  ISX_REQUIRE(HW >= 2, "isx_bn_stats_masked_fwd: unbiased std needs at least 2 pixels");
  ISX_CHECK_CUDA(cudaMemsetAsync(sums, 0, static_cast<size_t>(B) * C * 2 * sizeof(double), S(stream)));
  int rc = chan_sums(P(feat), B, HW, C, sums, S(stream), m, mask_b);
  if (rc) return rc;
  return bn_finalize(sums, B, C, HW, mean, std_, nullptr, nullptr, 1, 0.0, 0.0, nullptr, nullptr, nullptr, S(stream));
}

extern "C" int isx_mask_features(const isx_bf16* feat, const float* m, int mask_b, isx_bf16* fm, isx_bf16* fm2, int B,
                                 int64_t HW, int C, isx_stream stream) {
  ISX_REQUIRE(feat && m && fm && C % 8 == 0, "isx_mask_features: bad arguments");
  ISX_REQUIRE(mask_b == 1 || mask_b == B, "isx_mask_features: mask batch %d must be 1 or %d", mask_b, B);
  return mask_features(P(feat), m, mask_b, P(fm), P(fm2), B, HW, C, S(stream));
}

extern "C" int isx_avgpool2x2_f32(const float* in, float* out, int B, int H, int W, isx_stream stream) {
  ISX_REQUIRE(in && out && H >= 2 && W >= 2, "isx_avgpool2x2_f32: bad arguments");
  return avgpool2x2_f32(in, out, B, H, W, S(stream));
}

extern "C" int isx_tap_add_mask(const isx_bf16* g, const isx_bf16* add, const float* aff_a, const float* aff_b,
                                const isx_bf16* act, isx_bf16* out, int B, int64_t HW, int C, isx_stream stream) {
  ISX_REQUIRE(act && out, "isx_tap_add_mask: null pointer");
  return tap_add_mask(P(g), P(add), aff_a, aff_b, P(act), P(out), B, HW, C, S(stream));
}

// the option names of isx_set_option / isx_get_option and the context fields they address; nullptr: unknown name
static int IsxContext::*option_field(const char* name) {
  static const struct {
    const char* name;
    int IsxContext::*field;
  } kOptions[] = {
      {"c64", &IsxContext::opt_c64},
      {"halo2", &IsxContext::opt_halo2},
      {"tail_n", &IsxContext::opt_tail_n},
      {"sweep64", &IsxContext::opt_sweep64},
      {"smem_reserve_kb", &IsxContext::opt_smem_reserve_kb},
  };
  for (const auto& o : kOptions)
    if (strcmp(name, o.name) == 0) return o.field;
  return nullptr;
}

extern "C" int isx_set_option(const char* name, int value) {
  ISX_REQUIRE(name != nullptr, "isx_set_option: null name");
  int IsxContext::*field = option_field(name);
  ISX_REQUIRE(field != nullptr, "isx_set_option: unknown option '%s'", name);
  isx_ctx()->*field = value;
  return 0;
}

extern "C" int isx_get_option(const char* name, int* value) {
  ISX_REQUIRE(name != nullptr && value != nullptr, "isx_get_option: null pointer");
  int IsxContext::*field = option_field(name);
  ISX_REQUIRE(field != nullptr, "isx_get_option: unknown option '%s'", name);
  *value = isx_ctx()->*field;
  return 0;
}
