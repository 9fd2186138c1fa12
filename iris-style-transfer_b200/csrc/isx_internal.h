// Internal (C++) interfaces between the translation units of libisx.  The public C-ABI is
// include/isx.h; everything here is implementation detail.
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace isx {

struct ConvArgs {
  const __nv_bfloat16* in = nullptr;      // [B,H,W,Cin]
  const __nv_bfloat16* weight = nullptr;  // [ntaps][Cout][Cin] (x B when per_image_weights)
  __nv_bfloat16* out = nullptr;           // [B,H,W,Cout]
  int B = 0, H = 0, W = 0, Cin = 0, Cout = 0, ntaps = 9;
  // 1 or 2 (generic kernel only): out is [B, ceil(H/stride), ceil(W/stride), Cout], pixel (x, y) reads input
  // (stride*x + kx - 1, stride*y + ky - 1) for the 3x3 taps and (stride*x, stride*y) for ntaps = 1
  int stride = 1;
  bool per_image_weights = false;
  const float* bias = nullptr;
  int relu = 0;
  __nv_bfloat16* pool_out = nullptr;  // also write MaxPool2d(2,2)(out) [B,H/2,W/2,Cout] (fused into the epilogue when possible)
  // with pool_out: one routing byte per pooled element for the fused max-pool + ReLU backward (pool4_codes) [B,H/2,W/2,Cout]
  uint8_t* pool_idx = nullptr;
  // with pool_out + pool_idx: do not store the full-resolution output at all (nobody reads it: the backward routes through
  // pool_idx).  Honoured when the pool is fused into the epilogue; `out` must still be a valid buffer (fallback path).
  bool skip_out = false;
  const __nv_bfloat16* mask_act = nullptr;
  const __nv_bfloat16* add_buf = nullptr;
  const float* aff_a = nullptr;
  const float* aff_b = nullptr;
  int force_bn = 0, force_mt = 0, force_stages = 0;  // tuning / test hooks (0 = heuristic)
  // generic kernel only: the specialised 3x3 kernels sum in another order and are picked by the batch size, so a caller
  // whose results must not depend on the batch (ResNet-50 features: image i of a batch == image i alone) skips them
  bool generic_only = false;
  // fused Gram backward: out += gram_act . gram_D[b]   (gram_act [B,H,W,Cout], gram_D bf16 [B,Cout,Cout])
  const __nv_bfloat16* gram_act = nullptr;
  const __nv_bfloat16* gram_D = nullptr;
  // image-gradient tail (conv1_1 dgrad): when dx_nchw != null the epilogue writes fp32 NCHW instead of `out`
  float* dx_nchw = nullptr;
  int xc = 3;
  const float* in_mask = nullptr;
  int mask_b = 0;
};
int conv_tc(const ConvArgs& a, cudaStream_t stream);
bool conv_c64_applicable(const ConvArgs& a);
int conv_c64(const ConvArgs& a, cudaStream_t stream);
// Cin = Cout = 64 as a sweep with the sweep-axis taps stacked in N (conv_sweep.cu)
bool conv_sweep_applicable(const ConvArgs& a);
double conv_sweep_efficiency(const ConvArgs& a);
int conv_sweep(const ConvArgs& a, cudaStream_t stream);
// image-gradient tail with the taps in N (conv1_1_tail.cu)
int conv1_1_tail_n(const __nv_bfloat16* dy, const __nv_bfloat16* wd, const float* mask, int mask_b, float* dx, int xc,
                   int B, int H, int W, cudaStream_t stream);
// halo-patch kernel for the mid layers (conv_halo.cu)
bool conv_halo_applicable(const ConvArgs& a);
double conv_halo_efficiency(const ConvArgs& a);
int conv_halo(const ConvArgs& a, cudaStream_t stream);

// Gram partial products: partial[b][split][C][C] (fp32) = sum over the split's pixels of F^T F.
int gram_tc_partial(const __nv_bfloat16* feat, int B, int HW, int C, int splits, float* partial,
                    cudaStream_t stream);
int gram_pick_splits(int B, int HW, int C);
// mask-weighted variant (row G'): Gram of F * m with m fp32 [mask_b,HW]; kb_flags from gram_mask_flags; fm2 <- F * m^2 on
// the K blocks whose mask is not all zero (the caller zeroes fm2 once: untouched blocks must read as zero)
struct GramMask {
  const float* m;
  int mask_b;
  const uint8_t* kb_flags;
  __nv_bfloat16* fm2;
};
// csum (optional, C <= 128): fp32 [B][splits][C] per-channel sums of the features, computed by the tensor core alongside
int gram_sym_partial(const __nv_bfloat16* feat, int B, int HW, int C, int splits, float* partial, const GramMask* mask,
                     cudaStream_t stream, float* csum = nullptr);
int gram_mask_flags_bytes(int mask_b, int HW, int C);
int gram_mask_flags(const float* m, int mask_b, int HW, int C, uint8_t* flags, cudaStream_t stream);

}  // namespace isx
