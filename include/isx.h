/* libisx -- B200 (sm_100a) kernels for the iris-masked neural-style-transfer hot path of
 * AnonymWriter/Iris-Style-Transfer.  C ABI: plain device pointers, explicit shapes, a cudaStream_t;
 * every function returns 0 on success and != 0 on failure (text via isx_last_error()).  Nothing
 * here allocates device memory: the caller (e.g. a framework's caching allocator) owns every buffer,
 * including workspaces whose size is queried first.  Thread-compatible; no process-global mutable state (see isx_create).
 *
 * The reference has no FFI/plugin layer (it is pure Python): each entry point names the reference
 * call site (relative to the reference repo root) whose library kernels it replaces.
 *
 * Layouts: activations / gradients are NHWC bf16 ("isx_bf16" = 2-byte bfloat16), images and
 * image gradients are NCHW fp32 exactly as the reference passes them, Gram matrices [B,C,C] fp32.
 */
#ifndef ISX_H_
#define ISX_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ISX_VERSION 100

typedef uint16_t isx_bf16;   /* storage type of a bfloat16 */
typedef void* isx_stream;    /* cudaStream_t */

/* ---- status ------------------------------------------------------------------------------- */
const char* isx_last_error(void);
int isx_version(void);
/* fails unless `device` is an sm_100 part: there is no fallback path */
int isx_device_check(int device);

/* ---- peer memory over NVLink (one process per GPU of one box) ---------------------------------------------------------
 * isx_ipc_export: 64-byte handle of the cudaMalloc allocation that contains `ptr` + the byte offset of `ptr` inside it;
 * isx_ipc_open (in ANOTHER process of the box): maps that allocation into the caller's address space with peer access
 * enabled and returns its base; isx_ipc_close unmaps it.  Used by sharding.PeerRows: every rank pushes its feature rows
 * straight into every other rank's matrix (BASELINE config 3) with copy-engine copies instead of an all-gather kernel. */
int isx_ipc_export(const void* ptr, void* handle64, int64_t* offset);
int isx_ipc_open(const void* handle64, void** base_out);
int isx_ipc_close(void* base);
/* device-to-device copy on `stream` (cudaMemcpyAsync: copy engines); dst may be peer memory mapped with isx_ipc_open */
int isx_copy_d2d_async(void* dst, const void* src, int64_t bytes, isx_stream stream);

/* ---- handles ---------------------------------------------------------------------------------
 * The library keeps NO process-global mutable state.  Kernel-selection options (isx_set_option), the launch counter, the
 * CUDA-event profiler and the device's SM count (grid sizing) live in a context.  isx_create makes one for `device`,
 * isx_make_current binds it to the CALLING THREAD (NULL unbinds), isx_destroy frees it; every other entry point works on
 * the calling thread's current context.  A thread that never binds a handle gets a private default context (device = its
 * current CUDA device at first use), so single-threaded hosts -- the reference is one Python thread on one stream,
 * SURVEY.md §8b -- need no handle at all.  Thread-compatible: distinct threads may use distinct handles concurrently. */
typedef void* isx_handle;
int isx_create(int device, isx_handle* out);
int isx_destroy(isx_handle h);
int isx_make_current(isx_handle h);
int isx_sm_count(void);   /* SM count the current context sizes its grids with */

/* ---- weights: torchvision vgg19.features Conv2d parameters (models/vgg/vgg.py:43-49) ---------
 * fp32 OIHW [Cout,Cin,3,3] -> bf16 [9][Cout][Cin] for the forward conv and the 180-degree-rotated,
 * transposed [9][Cin][Cout] for dgrad.  Either output may be NULL. */
int isx_pack_conv3x3_weights(const float* w_oihw, int Cout, int Cin, isx_bf16* w_fwd, isx_bf16* w_dgrad,
                             isx_stream stream);

/* ---- K0+K1 head: Normalize -> [*mask] -> conv1_1 + bias + ReLU (models/vgg/vgg.py:81-87) ------
 * x: fp32 [B,xc,H,W], xc in {1,3} (1 broadcasts like transforms.Normalize does, SURVEY N3);
 * mask: NULL or fp32 [mask_b,1,H,W] with mask_b in {1,B}; w: fp32 [64,3,3,3]; out: bf16 [B,H,W,64]. */
int isx_conv1_1_fwd(const float* x, int xc, const float* mask, int mask_b, const float* w, const float* bias,
                    isx_bf16* out, int B, int H, int W, isx_stream stream);
/* Same head on the tensor cores: per-pixel 27-tap gather, bf16 hi+lo split of the normalised input (K = 64),
 * one tcgen05 128x64x64 MMA per 128 pixels.  w0_fwd: bf16 [64][64] from isx_pack_conv1_1_fwd. */
int isx_pack_conv1_1_fwd(const float* w, isx_bf16* w0_fwd, isx_stream stream);
int isx_conv1_1_fwd_tc(const float* x, int xc, const float* mask, int mask_b, const isx_bf16* w0_fwd, const float* bias,
                       isx_bf16* out, int B, int H, int W, isx_stream stream);
/* autograd tail of the same (pipelines.py:90): dY bf16 [B,H,W,64] (already ReLU-masked) ->
 * d(loss)/dx fp32 [B,xc,H,W], including Normalize's 1/std and the optional mask. */
int isx_conv1_1_dgrad(const isx_bf16* dy, const float* w, const float* mask, int mask_b, float* dx, int xc, int B,
                      int H, int W, isx_stream stream);

/* Same tail on the tensor cores: the 64->3 dgrad as a tcgen05 implicit GEMM with N padded to 16
 * (w0_dgrad: bf16 [9][16][64] from isx_pack_conv1_1_dgrad) and an fp32-NCHW epilogue. */
int isx_pack_conv1_1_dgrad(const float* w, isx_bf16* w0_dgrad, isx_stream stream);
int isx_conv1_1_dgrad_tc(const isx_bf16* dy, const isx_bf16* w0_dgrad, const float* mask, int mask_b, float* dx, int xc,
                         int B, int H, int W, isx_stream stream);

/* ---- K1: Conv2d 3x3 s1 p1 + bias + ReLU on tcgen05 (models/vgg/vgg.py:87) ---------------------
 * in bf16 [B,H,W,Cin], w_fwd from isx_pack_conv3x3_weights, bias fp32 [Cout], out bf16 [B,H,W,Cout].
 * Cin, Cout multiples of 64.  tile_cfg: 0 = heuristic, else BN*100 + MT*10 + stages (test / tuning hook). */
int isx_conv3x3_bias_relu_fwd(const isx_bf16* in, const isx_bf16* w_fwd, const float* bias, isx_bf16* out, int B,
                              int H, int W, int Cin, int Cout, int relu, int tile_cfg, isx_stream stream);

/* K1 + K2 fused: same conv, and MaxPool2d(2,2) of its ReLU output written to pool_out bf16 [B,H/2,W/2,Cout] from the
 * epilogue's staged tile (falls back to a separate pool launch when the pixel patch has an odd side). */
int isx_conv3x3_bias_relu_pool_fwd(const isx_bf16* in, const isx_bf16* w_fwd, const float* bias, isx_bf16* out,
                                   isx_bf16* pool_out, int B, int H, int W, int Cin, int Cout, int tile_cfg,
                                   isx_stream stream);
/* The same, and the ROUTING BYTES of the pool's backward: pool_idx uint8 [B,H/2,W/2,Cout], one byte per pooled element --
 * 0..3 = window position (0,0),(0,1),(1,0),(1,1) of the FIRST maximum (ATen's rule), 4 = the maximum is <= 0, i.e. the ReLU
 * passes nothing.  isx_maxpool2x2_bwd_idx then needs the pooled gradient and these bytes only, not the pre-pool activation
 * (autograd of MaxPool2d + ReLU, pipelines.py:90).  skip_out != 0: the full-resolution output is not stored at all when the
 * pool is fused into the epilogue (`out` must still point to a [B,H,W,Cout] buffer: the unfused fallback writes it). */
int isx_conv3x3_bias_relu_pool_idx_fwd(const isx_bf16* in, const isx_bf16* w_fwd, const float* bias, isx_bf16* out,
                                       isx_bf16* pool_out, uint8_t* pool_idx, int skip_out, int B, int H, int W, int Cin,
                                       int Cout, int tile_cfg, isx_stream stream);

/* ---- K3: conv dgrad (+ tap gradient, x ReLU mask) on tcgen05 (loss.backward(), pipelines.py:90)
 * dy bf16 [B,H,W,Cout] -> dx bf16 [B,H,W,Cin] for the forward conv Cin->Cout; weights frozen so
 * there is no wgrad (models/vgg/vgg.py:52-53).  Epilogue, all optional:
 *   dx += add_grad[B,H,W,Cin]                      (Gram tap gradient of the layer below)
 *   dx += aff_a[b,c] + aff_b[b,c]*act              (BN-statistics tap gradient; needs relu_act)
 *   dx  = relu_act > 0 ? dx : 0                    (ReLU backward of the layer below) */
int isx_conv3x3_dgrad(const isx_bf16* dy, const isx_bf16* w_dgrad, isx_bf16* dx, int B, int H, int W, int Cin,
                      int Cout, const isx_bf16* relu_act, const isx_bf16* add_grad, const float* aff_a,
                      const float* aff_b, int tile_cfg, isx_stream stream);

/* K3 + K5 fused: dx = relu'(act_below) * (dgrad(dy) + act_below . D[b]) -- the Gram tap gradient of the layer below
 * (gram_D bf16 [B,Cin,Cin] from isx_gram_fwd) rides the same tcgen05 main loop as Cin/64 extra K blocks. */
int isx_conv3x3_dgrad_gram(const isx_bf16* dy, const isx_bf16* w_dgrad, isx_bf16* dx, int B, int H, int W, int Cin,
                           int Cout, const isx_bf16* act_below, const isx_bf16* gram_D, isx_stream stream);

/* ---- K2: MaxPool2d(2,2) fwd / bwd (bwd fused with the ReLU mask of the pre-pool activation) ---- */
int isx_maxpool2x2_fwd(const isx_bf16* in, isx_bf16* out, int B, int H, int W, int C, isx_stream stream);
int isx_maxpool2x2_bwd(const isx_bf16* dy_pooled, const isx_bf16* act_prepool, isx_bf16* dx, int B, int H, int W,
                       int C, isx_stream stream);
/* the same pair through routing bytes (see isx_conv3x3_bias_relu_pool_idx_fwd): fwd writes out (may be NULL) and idx uint8
 * [B,H/2,W/2,C]; bwd reads 3 bytes per pooled element instead of the four pre-pool activations */
int isx_maxpool2x2_fwd_idx(const isx_bf16* in, isx_bf16* out, uint8_t* idx, int B, int H, int W, int C, isx_stream stream);
int isx_maxpool2x2_bwd_idx(const isx_bf16* dy_pooled, const uint8_t* idx, isx_bf16* dx, int B, int H, int W, int C,
                           isx_stream stream);

/* ---- K4: Gram matrix (utils.py:242-257 GramMatrix) ---------------------------------------------
 * feat bf16 [B,HW,C] (NHWC flattened), C in {64,128,256,512}.  G = F^T F * inv_n (fp32 [B,C,C]).
 * workspace: isx_gram_workspace_bytes(B,HW,C) bytes.  With a target (fp32 [target_b,C,C],
 * target_b in {1,B}): loss[b] += loss_scale * sum((G-T)^2) (double, caller zeroes) and
 * D = grad_scale * (G - T) in bf16 [B,C,C] for isx_gram_bwd.  G_out / target / loss / D may be NULL. */
int64_t isx_gram_workspace_bytes(int B, int HW, int C);
int isx_gram_fwd(const isx_bf16* feat, int B, int HW, int C, float inv_n, void* workspace, float* G_out,
                 const float* target, int target_b, double loss_scale, double* loss, float grad_scale,
                 isx_bf16* D_out, isx_stream stream);
/* Mask-weighted Gram (row G' of the hot path; hooks models/vgg/vgg.py:84-85, pipelines.py:83): G = (F*m)^T (F*m) * inv_n
 * with m fp32 [mask_b,HW], mask_b in {1,B}.  The weights are applied to the operand tiles inside the Gram kernel and K
 * blocks whose mask is all zero are skipped.  flags_ws: isx_gram_mask_flags_bytes(mask_b,HW,C) bytes of scratch;
 * fm2 (bf16 [B,HW,C], required) receives F*m^2, the operand of the Gram backward (dF = (F m^2) . D): written on the
 * non-zero blocks, zeroed elsewhere.  Other arguments as isx_gram_fwd. */
int64_t isx_gram_mask_flags_bytes(int mask_b, int HW, int C);
int isx_gram_masked_fwd(const isx_bf16* feat, int B, int HW, int C, const float* m, int mask_b, void* flags_ws,
                        isx_bf16* fm2, float inv_n, void* workspace, float* G_out, const float* target, int target_b,
                        double loss_scale, double* loss, float grad_scale, isx_bf16* D_out, isx_stream stream);
/* ---- K5: Gram backward dF[b] = F[b] . D[b] (autograd of utils.py:253-256), tcgen05 1x1 mode.
 * feat bf16 [B,H,W,C], D bf16 [B,C,C] (symmetric), dF bf16 [B,H,W,C]; optional relu mask. */
int isx_gram_bwd(const isx_bf16* feat, const isx_bf16* D, isx_bf16* dF, int B, int H, int W, int C,
                 const isx_bf16* relu_act, isx_stream stream);

/* ---- K6: content MSE (utils.py:285-290) and mean/std statistics (utils.py:337-354, classifiers.py:71)
 * content: loss[b] += loss_scale * sum((p-t)^2); grad = grad_scale*(p-t)*(p>0) (bf16, may be NULL). */
int isx_content_mse_fwd_bwd(const isx_bf16* pred, const isx_bf16* target, int target_b, isx_bf16* grad, int B,
                            int64_t per_image, double loss_scale, float grad_scale, double* loss, isx_stream stream);
/* the same without the fused ReLU backward when relu_mask == 0: grad = grad_scale*(p-t) (autograd of F.mse_loss, utils.py:288) */
int isx_mse_fwd_bwd(const isx_bf16* pred, const isx_bf16* target, int target_b, isx_bf16* grad, int B, int64_t per_image,
                    double loss_scale, float grad_scale, int relu_mask, double* loss, isx_stream stream);
/* out[b,p,c] = a[b,c] + b[b,c] * feat[b,p,c]  [* (feat > 0)]: the backward of per-channel mean / std statistics
 * (autograd of utils.py:337-338 / classifiers.py:71) is affine in the feature map */
int isx_channel_affine(const isx_bf16* feat, const float* a, const float* b, isx_bf16* out, int B, int64_t HW, int C,
                       int relu_mask, isx_stream stream);
/* sums: double [B,C,2] workspace.  mean/std fp32 [B,C] (std unbiased).  With targets: loss[b] +=
 * loss_scale * sum_c[(mu-mu_t)^2+(sd-sd_t)^2] and affine tap-gradient coefficients aff_a/aff_b [B,C]. */
int isx_bn_stats_fwd(const isx_bf16* feat, int B, int64_t HW, int C, double* sums, float* mean, float* std_,
                     const float* t_mean, const float* t_std, int target_b, double loss_scale, double grad_scale,
                     double* loss, float* aff_a, float* aff_b, isx_stream stream);
/* mean / unbiased std of the MASK-WEIGHTED features F * m (m fp32 [mask_b,HW]): targets of the mask-weighted BN loss */
int isx_bn_stats_masked_fwd(const isx_bf16* feat, const float* m, int mask_b, int B, int64_t HW, int C, double* sums, float* mean,
                            float* std_, isx_stream stream);
/* ---- G' (extension; hooks models/vgg/vgg.py:84-85, pipelines.py:83): mask-weighted Gram input.  fm = feat * m,
 * fm2 = feat * m^2 (optional) with m fp32 [mask_b,HW] the iris mask at the layer's resolution; the mask pyramid is
 * m_{l+1} = 2x2 average pool of m_l (isx_avgpool2x2_f32).  Gram(fm) == utils.GramMatrix(F * m_l). */
int isx_mask_features(const isx_bf16* feat, const float* m, int mask_b, isx_bf16* fm, isx_bf16* fm2, int B, int64_t HW,
                      int C, isx_stream stream);
int isx_avgpool2x2_f32(const float* in, float* out, int B, int H, int W, isx_stream stream);
/* out = (g + add + aff) * (act > 0) -- tap gradient at a layer that no dgrad epilogue feeds; g/add/aff may be NULL */
int isx_tap_add_mask(const isx_bf16* g, const isx_bf16* add, const float* aff_a, const float* aff_b,
                     const isx_bf16* act, isx_bf16* out, int B, int64_t HW, int C, isx_stream stream);

/* ---- K7/K8: torch.optim.LBFGS([x], lr) with defaults (pipelines.py:59,103; torch/optim/lbfgs.py:333-537)
 * P independent problems of N floats each advance in lock step, one closure evaluation per tick.
 * All optimiser scalars live in device memory (state: isx_lbfgs_state_bytes(P)); history S,Y:
 * fp32 (or bf16, cfg->history_bf16) [P][history+1][N] each; mats: isx_lbfgs_mats_bytes(P, history); scratch: isx_lbfgs_scratch_bytes. */
typedef struct {
  int32_t epochs;            /* closure evaluations requested (pipelines.py:16,79) */
  int32_t max_iter;          /* 20 */
  int32_t max_eval;          /* 25 */
  int32_t history;           /* 100 (<= 100) */
  int32_t history_bf16;      /* 0: S,Y fp32 like the reference; 1: bf16 (halves the traffic of both history passes) */
  int32_t reserved_;
  double lr;                 /* 1.0 */
  double tolerance_grad;     /* 1e-7 */
  double tolerance_change;   /* 1e-9 */
  double c_weight, s_weight; /* alpha, beta of pipelines.py:89 */
} isx_lbfgs_config;
int64_t isx_lbfgs_state_bytes(int P);
int64_t isx_lbfgs_mats_bytes(int P, int history);
int64_t isx_lbfgs_scratch_bytes(int P, int64_t N, int history);
int isx_lbfgs_init(void* state, int P, isx_stream stream);
/* One tick AFTER a closure evaluation produced grad and the per-image losses:
 * memory update + direction + x = clamp(x + t d, 0, 1) (lbfgs.py:396-526 + pipelines.py:82), or the
 * early-exit bookkeeping.  loss_c/loss_s: double [P*images_per_problem]; hist_c/hist_s: double
 * [evaluations][P] loss logs (pipelines.py:94-95), row = the problem's own evaluation counter (`tick` is
 * informational: every launch parameter is tick-invariant so one tick can be captured in a CUDA graph). */
int isx_lbfgs_tick(float* x, const float* grad, float* grad_prev, void* S, void* Y, void* state, void* mats,
                   void* scratch, const double* loss_c, const double* loss_s, int images_per_problem, int P,
                   int64_t N, const isx_lbfgs_config* cfg, double* hist_c, double* hist_s, int tick,
                   isx_stream stream);
/* isx_lbfgs_tick with per-problem loss weights: problem p's loss (its tolerance_change test) is
 * c_weight[p] * c_p + s_weight[p] * s_p with c_weight / s_weight device double [P]; cfg->c_weight / s_weight are not read. */
int isx_lbfgs_tick_problems(float* x, const float* grad, float* grad_prev, void* S, void* Y, void* state, void* mats,
                            void* scratch, const double* loss_c, const double* loss_s, int images_per_problem, int P,
                            int64_t N, const isx_lbfgs_config* cfg, const double* c_weight, const double* s_weight,
                            double* hist_c, double* hist_s, int tick, isx_stream stream);
/* done_out[p] (device int32) <- number of closure evaluations problem p performed once it has finished its
 * pipelines.py:79 loop, 0 while it is still running */
int isx_lbfgs_done_flags(const void* state, int P, int32_t* done_out, isx_stream stream);
/* count_out[p] (device int32) <- number of (y, s) pairs problem p currently holds in its history ring (len(old_dirs),
 * lbfgs.py:409-417): what the two history passes of the next tick will stream */
int isx_lbfgs_history_counts(const void* state, int P, int32_t* count_out, isx_stream stream);
int isx_clamp01(float* x, int64_t n, isx_stream stream);

/* ---- fused driver: one closure evaluation of pipelines.py:80-91 ------------------------------- */
#define ISX_MAX_TAPS 8
#define ISX_VGG19_CONVS 16
#define ISX_TAP_POOL0 16       /* tap ids: 0..15 = ReLU output of conv i; 16..20 = output of MaxPool 0..4 (pool1..pool5) */
#define ISX_VGG19_TAPS 21
typedef struct {
  int32_t B, H, W, xc;                  /* image batch fp32 [B,xc,H,W] */
  int32_t n_conv;                       /* number of convs to run (deepest tapped conv index + 1) */
  int32_t style_mode;                   /* 0: Gram (utils.StyleLoss_Gram), 1: mean/std (utils.StyleLoss_BN) */
  int32_t n_style;
  int32_t style_conv[ISX_MAX_TAPS];     /* tap id: conv index (0..15) whose ReLU output is tapped, or ISX_TAP_POOL0 + k */
  float style_w[ISX_MAX_TAPS];
  int32_t n_content;
  int32_t content_conv[ISX_MAX_TAPS];
  float content_w[ISX_MAX_TAPS];
  int32_t style_target_b;               /* 1 or B */
  int32_t content_target_b;             /* 1 or B */
  int32_t coupled;                      /* 1: batch is ONE problem -> content loss is a mean over the batch too */
  int32_t mask_b;                       /* 0: no input mask, else 1 or B */
  int32_t style_mask_b;                 /* 0: plain losses; 1 or B: mask-weighted style loss (row G': Gram or BN statistics of F * m_l) */
  int32_t pred_unbatched;               /* 1: the content image was passed UNBATCHED (3,H,W): utils.GramMatrix then divides the
                                           prediction's Gram by H*W instead of C*H*W (utils.py:253-254, n = x[0].numel()) */
  double c_weight, s_weight;            /* alpha, beta */
} isx_nst_config;

typedef struct {
  const float* w0;                      /* conv1_1 fp32 OIHW [64,3,3,3] */
  const isx_bf16* w0_fwd;               /* isx_pack_conv1_1_fwd (tensor-core head); NULL -> CUDA-core head */
  const isx_bf16* w0_dgrad;             /* isx_pack_conv1_1_dgrad (tensor-core image-gradient tail); NULL -> CUDA-core tail */
  const float* bias[ISX_VGG19_CONVS];   /* fp32 [Cout] per conv */
  const isx_bf16* w_fwd[ISX_VGG19_CONVS];    /* packed (isx_pack_conv3x3_weights); [0] unused */
  const isx_bf16* w_dgrad[ISX_VGG19_CONVS];
  void* workspace;                      /* isx_nst_workspace_bytes(cfg) */
  const isx_bf16* content_target[ISX_MAX_TAPS];  /* bf16 NHWC [content_target_b,h,w,C] */
  const float* gram_target[ISX_MAX_TAPS];        /* fp32 [style_target_b,C,C] */
  const float* bn_target_mean[ISX_MAX_TAPS];     /* fp32 [style_target_b,C] */
  const float* bn_target_std[ISX_MAX_TAPS];
  const float* input_mask;              /* fp32 [mask_b,1,H,W] or NULL (VGG19.forward(x, mask), vgg.py:84-85) */
  const float* style_mask[ISX_MAX_TAPS];/* fp32 [style_mask_b,h_l,w_l]: iris mask at each style layer's resolution (G') */
} isx_nst_buffers;

int64_t isx_nst_workspace_bytes(const isx_nst_config* cfg);
/* autograd of VGG19.forward alone (pipelines.py:90 when the caller owns the loss): feat_grads has ISX_VGG19_TAPS entries,
 * feat_grads[id] = bf16 NHWC gradient w.r.t. tap id (ReLU output of conv id, or pool id - 16; NULL where none),
 * last_pool_grad = gradient w.r.t. the pool after the deepest conv
 * (or NULL); uses the activations the preceding isx_nst_forward left in the workspace; grad fp32 [B,xc,H,W]. */
int isx_nst_backward(const isx_nst_config* cfg, const isx_nst_buffers* bufs, const isx_bf16* const* feat_grads,
                     const isx_bf16* last_pool_grad, float* grad, isx_stream stream);
/* forward only (VGG19.forward, models/vgg/vgg.py:69-92) up to conv index n_conv-1; activations stay in the workspace, see
 * isx_nst_feature.  flags: ISX_FWD_LAST_POOL = also the pool after the deepest conv; ISX_FWD_LEAN = a pre-pool ReLU output
 * that is not a tap is NOT materialised (only its pooled map and the routing bytes of the pool's backward are written:
 * isx_nst_backward and isx_nst_style_features never read it; isx_nst_feature(kind 0) of such a conv is then undefined). */
#define ISX_FWD_LAST_POOL 1
#define ISX_FWD_LEAN 2
int isx_nst_forward(const isx_nst_config* cfg, const isx_nst_buffers* bufs, const float* x, int flags,
                    isx_stream stream);
/* device pointer / shape of a stored activation: kind 0 = ReLU output of conv `idx`, 1 = output of pool `idx` (0..4) */
int isx_nst_feature(const isx_nst_config* cfg, const isx_nst_buffers* bufs, int kind, int idx, isx_bf16** ptr,
                    int32_t* h, int32_t* w, int32_t* c);
/* row G': call once after the style masks (bufs->style_mask) were set or changed and before isx_nst_eval: zeroes the
 * F * m^2 buffers of the workspace and records which K blocks of every mask are non-zero (the Gram kernel skips the
 * others: an iris mask covers 6-10 % of an eye frame) */
int isx_nst_prepare_style_masks(const isx_nst_config* cfg, const isx_nst_buffers* bufs, isx_stream stream);
/* style features of the batch the preceding isx_nst_forward left in the workspace, one row per image written straight
 * into out (row stride ld floats): [per style tap: mean | unbiased std over (H,W)] (models/classifiers/classifiers.py:71)
 * then [per style tap: upper triangle of utils.GramMatrix in torch.triu_indices order] (BASELINE config 3) */
int isx_nst_style_features(const isx_nst_config* cfg, const isx_nst_buffers* bufs, int want_stats, int want_gram,
                           float* out, int64_t ld, isx_stream stream);
/* closure evaluation: loss_c/loss_s double [B] (unweighted, per image), grad fp32 [B,xc,H,W] = d(alpha c + beta s)/dx */
int isx_nst_eval(const isx_nst_config* cfg, const isx_nst_buffers* bufs, const float* x, double* loss_c,
                 double* loss_s, float* grad, isx_stream stream);

/* ---- several coupled problems in one batch: P = B / g problems of g images each (nst(problem_size=g)) ---------------
 * Problem p is the images [p*g, (p+1)*g): its content loss is the mean over its g images, its style loss the sum, and it
 * has its own alpha / beta.  The weights are read from device memory on every call, so a captured tick stays valid. */
typedef struct {
  int32_t images_per_problem;           /* g >= 1, B % g == 0 */
  int32_t style_target_b;               /* 1, P or B: image b reads style target b / (B / style_target_b); replaces
                                           cfg->style_target_b */
  const double* c_weight;               /* device [P]: alpha of each problem (cfg->c_weight is not read) */
  const double* s_weight;               /* device [P]: beta of each problem (cfg->s_weight is not read) */
} isx_nst_problems;
/* isx_nst_eval for P problems: same outputs (per-image unweighted losses), grad = d(sum_p alpha_p c_p + beta_p s_p)/dx.
 * cfg->coupled is not read.  With g = B, style_target_b in {1, B} and equal weights this is isx_nst_eval with coupled = 1,
 * with g = 1 isx_nst_eval with coupled = 0, bit for bit. */
int isx_nst_eval_problems(const isx_nst_config* cfg, const isx_nst_buffers* bufs, const isx_nst_problems* problems,
                          const float* x, double* loss_c, double* loss_s, float* grad, isx_stream stream);

/* ---- K10: iris mask + bounding box (pipelines.py:139-165 mask_and_crop_iris; utils.py:44-72 crop_image) --
 * x fp32 [B,1,H,W]; seg int64 [B,1,H,W] label map or NULL; m = (seg == label) & (x <= threshold) (either
 * test can be off: seg NULL / use_threshold 0); mask uint8 [B,1,H,W] (0/1) and xm = x*m are optional
 * outputs; bbox int32 [B,4] = (x_min, y_min, x_max, y_max) = (row_min, col_min, row_max, col_max) of the
 * NONZERO PIXELS of x*m, inclusive (utils.py:57-64).  No nonzero pixel -> row_max = -1 (the reference
 * raises on the empty min()).  Bit-exact integer work. */
int isx_mask_bbox(const float* x, const int64_t* seg, int label, int use_threshold, float threshold, uint8_t* mask,
                  float* xm, int32_t* bbox, int B, int H, int W, isx_stream stream);
/* isx_mask_bbox for a label map of either dtype: seg_dtype 0 = int64 (= isx_mask_bbox), 1 = uint8 [B,1,H,W], compared as
 * int(seg) == label, so the result equals the int64 call on the widened map (a label outside 0..255 matches nothing).  Any
 * other seg_dtype is an error. */
int isx_mask_bbox_typed(const float* x, const void* seg, int seg_dtype, int label, int use_threshold, float threshold,
                        uint8_t* mask, float* xm, int32_t* bbox, int B, int H, int W, isx_stream stream);
/* torchvision v2 Resize (bilinear, antialias=True) of the window src_bbox (or the whole image when NULL) of
 * src fp32 [B,src_c,SH,SW] to dst fp32 [B,dst_c,DH,DW]; src_c == 3 is converted to gray first
 * (rgb_to_grayscale, …2019.py:112); the single result channel is replicated dst_c times (…2019.py:79). */
int isx_resize_bilinear_aa(const float* src, int src_c, int SH, int SW, const int32_t* src_bbox, float* dst, int dst_c,
                           int DH, int DW, int B, isx_stream stream);
/* …2019.py:64-79 / …2020.py:78-100 for a whole batch in one launch: (frame * mask)[bbox] -> Resize((DH,DW)) bilinear
 * antialiased -> replicated to dst_c channels.  frames fp32 [B,1,H,W], mask uint8 [B,1,H,W], bbox int32 [B,4] (ragged);
 * dst fp32 [B,dst_c,DH,DW] must be zero-initialised by the caller: a frame whose bbox is empty is left untouched. */
int isx_crop_resize_masked(const float* frames, const uint8_t* mask, const int32_t* bbox, float* dst, int dst_c, int DH,
                           int DW, int B, int H, int W, isx_stream stream);
/* ---- K9: composite (…2019.py:111-130, …2020.py:121-139): gray(new_iris) -> Resize(bbox shape) -> * mask ->
 * frames[bbox] = frames[bbox] * ~mask + new, in place.  new_iris fp32 [B,src_c,SH,SW], frames fp32 [B,1,H,W],
 * mask uint8 [B,1,H,W], bbox int32 [B,4]. */
int isx_composite(const float* new_iris, int src_c, int SH, int SW, float* frames, const uint8_t* mask,
                  const int32_t* bbox, int B, int H, int W, isx_stream stream);

/* ---- mask producer: RITnet (models/ritnet/ritnet.py:8-223; call sites iris_style_transfer_openeds2019.py:155,
 * data_preprocessing.py:165, pipelines.py:133-141) for a batch of frames in one call --------------------------------
 * x fp32 [B,1,H,W] in [0,1] (H, W multiples of 16) -> labels int64 [B,H,W] in {0,1,2,3} (2 = iris), optionally the logits
 * fp32 [B,4,H,W].  RITnet_transform (ritnet.py:79-98) runs on the device, bit-exact with the reference's OpenCV round trip:
 * gamma_lut = the 256 uint8 values np.uint8(255 * linspace(0,1,256)**0.8) (ritnet.py:72,93-94), norm_lut = the 256 floats
 * ToDtype(scale)/Normalize(0.5,0.5) map uint8 to (ritnet.py:73-77), CLAHE(clipLimit 1.5, 8x8 tiles) restated from OpenCV.
 * params: isx_ritnet_param_floats() floats = the DenseNet2D state dict in network order: per down block conv1, conv21,
 * conv22, conv31, conv32 (each weight as [kh*kw][Cin][32] then bias[32]) then the BatchNorm folded to scale[32], shift[32];
 * per up block conv11, conv12, conv21, conv22; then out_conv1 weight [4][32] and bias[4].  fp32 throughout. */
/* RITnet_transform alone (any H, W >= 8): x fp32 [B,1,H,W] -> out fp32 [B,1,H,W], the network's input */
int64_t isx_ritnet_transform_workspace_bytes(int B, int H, int W);
int isx_ritnet_transform(const float* x, const uint8_t* gamma_lut, const float* norm_lut, void* workspace, float* out, int B,
                         int H, int W, isx_stream stream);
int64_t isx_ritnet_param_floats(void);
int64_t isx_ritnet_workspace_bytes(int B, int H, int W);
int isx_ritnet_forward(const float* x, const float* params, const uint8_t* gamma_lut, const float* norm_lut, void* workspace,
                       int64_t* labels, float* logits, int B, int H, int W, isx_stream stream);
/* isx_ritnet_forward writing labels of label_dtype 0 = int64 (= isx_ritnet_forward) or 1 = uint8 [B,H,W] (same values, 1 B
 * per pixel); any other label_dtype is an error.  The logits do not depend on it. */
int isx_ritnet_forward_typed(const float* x, const float* params, const uint8_t* gamma_lut, const float* norm_lut,
                             void* workspace, void* labels, int label_dtype, float* logits, int B, int H, int W,
                             isx_stream stream);

/* ---- classifier heads (models/classifiers/classifiers.py:3-72; iris_classification.py:66-71, …2019.py:82-84) -----------
 * A Linear layer over a batch of M <= 256 eyes is a weight-streaming tcgen05 GEMM out^T[N,M] = W'[N,K'] . X'[M,K']^T with
 * K' = K + 64: column K of X' is 1 and column K of W' the bias (K a multiple of 64).  Packed operands are bf16:
 *   isx_linear_pack        fp32 W [N,K] (nn.Linear layout), bias [N] -> W' [Npad, K+64] (rows >= N zero), once per model
 *   isx_rows_pack          fp32 rows [M,K] (row stride ld_src)      -> X' [Mpad, K+64], Mpad a multiple of 64
 *   isx_pool7_flatten_pack pool5 bf16 NHWC [B,h,w,C] -> AdaptiveAvgPool2d(7,7) + Flatten (c*49+i*7+j) -> X' [Mpad, 49C+64]
 *   isx_linear_fwd         out^T bf16 [Npad, Mpad] = relu?(W' . X'^T)
 *   isx_transpose_pack     out^T [N, Mpad] -> the next layer's X' [Mpad, N+64]; isx_transpose_out -> fp32 logits [M, N] */
int isx_linear_pack(const float* W, const float* bias, int N, int K, int Npad, isx_bf16* dst, isx_stream stream);
int isx_rows_pack(const float* src, int64_t ld_src, int M, int K, int Mpad, isx_bf16* dst, isx_stream stream);
int isx_pool7_flatten_pack(const isx_bf16* pool5, int B, int h, int w, int C, int Mpad, isx_bf16* dst, isx_stream stream);
int isx_linear_fwd(const isx_bf16* Xp, const isx_bf16* Wp, isx_bf16* outT, int Mpad, int Npad, int Kp, int relu, isx_stream stream);
int isx_transpose_pack(const isx_bf16* srcT, int N, int Mpad, int M, isx_bf16* dst, isx_stream stream);
int isx_transpose_out(const isx_bf16* srcT, int N, int Mpad, int M, float* dst, isx_stream stream);

/* ---- downstream evaluator features (models/gaze_estimators/gaze_estimators.py) --------------------------------------------
 * isx_eye_landmarks = extract_eye_landmarks (gaze_estimators.py:108-178; call sites data_preprocessing.py:412,
 * gaze_estimators.py:49,291) for a BATCH of label maps in one call, without the reference's per-image `.cpu().numpy()` round
 * trip: cv2.findContours(RETR_EXTERNAL, CHAIN_APPROX_SIMPLE) -> max(contourArea) -> cv2.fitEllipse for the pupil (label 3) and
 * the iris (label 2) (:55-83), np.where min / max for the sclera (label 1) (:85-106), the derived ratios (:139-152).
 * seg [B,H,W], seg_dtype 0 = int64, 1 = uint8, 2 = int32 (compared after `.astype(np.uint8)` like :127); landmarks fp32
 * [B,19] in the order of :154-174, absent quantities 0 (:176); info int32 [B,8] (may be NULL) = {pupil: points of the chosen
 * contour, external contours, flags; iris: the same three; sclera present; 0}.  flags bit 0: the chosen contour has exactly
 * five points or a rank-deficient system -- there cv2.fitEllipse leaves the general algorithm (fitEllipseDirect / a
 * pseudo-random perturbation) and this library does not follow it: it solves the unperturbed system; bit 1: the contour has
 * more than max_points points (nothing fitted: call again with a larger workspace).  The reference asserts H, W = 400, 640;
 * any frame whose three padded bit planes fit in shared memory is accepted (3 * (H+2) * ceil((W+2)/32) * 4 <= 200 KB). */
int64_t isx_eye_landmarks_workspace_bytes(int B, int H, int W, int max_points);
int isx_eye_landmarks(const void* seg, int seg_dtype, int B, int H, int W, double epsilon, int max_points, void* workspace,
                      float* landmarks, int32_t* info, isx_stream stream);
/* GazeEstimator1.model / GazeEstimator2.model in eval mode + the row normalisation (gaze_estimators.py:24-32,51-53 and
 * :196-204,221-223): out[B,out_dim] = y / ||y||_2, y = W3 relu(W2 relu(W1 x + b1) + b2) + b3; fp32, torch.nn.Linear layouts
 * (W1 [hidden,in_dim], W2 [hidden,hidden], W3 [out_dim,hidden]); x fp32 rows with stride ld_x. */
int isx_gaze_head_fwd(const float* x, int64_t ld_x, int B, int in_dim, int hidden, int out_dim, const float* W1, const float* b1,
                      const float* W2, const float* b2, const float* W3, const float* b3, float* out, isx_stream stream);

/* ---- ResNet-50 trunk: the feature extractor of GazeEstimator2(extract_feature=True) (models/gaze_estimators/
 * gaze_estimators.py:180-223 over models/resnet/resnet.py = torchvision resnet50 without fc, eval mode) -------------------
 * Activations bf16 NHWC, fp32 accumulation.  BatchNorm is folded into every convolution beforehand (eval mode), so each
 * layer is conv + bias.  Output sizes round up like torchvision's: a stride-2 layer maps H to ceil(H / 2).
 * isx_conv_bias_act_fwd: in [B,H,W,Cin] -> out [B,ceil(H/stride),ceil(W/stride),Cout] = relu?(conv(in) + bias [+ residual]);
 *   k = 1 (pad 0; w from isx_pack_conv1x1_weights) or 3 (pad 1; w_fwd from isx_pack_conv3x3_weights), stride 1 or 2,
 *   Cin and Cout multiples of 64; residual (may be NULL) has out's shape and is added before the ReLU (Bottleneck.forward).
 * isx_pack_conv1x1_weights: fp32 [Cout,Cin(,1,1)] -> bf16 [Cout][Cin].
 * isx_resnet_stem_fwd: conv1 (7x7, stride 2, pad 3, 3 -> 64) + bias + ReLU, straight from the fp32 NCHW image
 *   x [B,xc,H,W] (xc = 1 broadcasts to three channels) -> bf16 [B,ceil(H/2),ceil(W/2),64]; w from
 *   isx_pack_resnet_stem_weights (fp32 OIHW [64,3,7,7] -> bf16 [64][192]).
 * isx_maxpool3x3s2_fwd: MaxPool2d(3, 2, padding 1) bf16 [B,H,W,C] -> [B,ceil(H/2),ceil(W/2),C], C a multiple of 8;
 *   bit-identical to torch (padding is -inf, the first maximum of the window wins, NaN propagates).
 * isx_global_avgpool: AdaptiveAvgPool2d(1) + flatten, bf16 [B,HW,C] -> fp32 [B,C]; C a multiple of 8; deterministic. */
int isx_pack_conv1x1_weights(const float* w, int Cout, int Cin, isx_bf16* w_out, isx_stream stream);
int isx_pack_resnet_stem_weights(const float* w, isx_bf16* w_out, isx_stream stream);
int isx_conv_bias_act_fwd(const isx_bf16* in, const isx_bf16* w, const float* bias, const isx_bf16* residual, isx_bf16* out,
                          int B, int H, int W, int Cin, int Cout, int k, int stride, int relu, isx_stream stream);
int isx_resnet_stem_fwd(const float* x, int xc, const isx_bf16* w, const float* bias, isx_bf16* out, int B, int H, int W,
                        isx_stream stream);
int isx_maxpool3x3s2_fwd(const isx_bf16* in, isx_bf16* out, int B, int H, int W, int C, isx_stream stream);
int isx_global_avgpool(const isx_bf16* in, float* out, int B, int HW, int C, isx_stream stream);
/* The whole trunk: x fp32 [B,xc,H,W] (xc in {1,3}, H and W >= 32, no input normalisation) -> feat_out fp32 [B,2048].
 * weights: the 53 folded (weight, bias) pairs in torchvision module order -- conv1, then per Bottleneck of layer1..layer4
 * conv1 (1x1), conv2 (3x3, carries the stride), conv3 (1x1), and after the first block's conv3 its downsample.0 (1x1,
 * strided).  w[0] from isx_pack_resnet_stem_weights, 1x1 from isx_pack_conv1x1_weights, 3x3 the w_fwd of
 * isx_pack_conv3x3_weights; bias fp32 [Cout].  workspace: isx_resnet50_workspace_bytes(B, H, W) bytes (host-only query;
 * -1 and isx_last_error for B < 1 or H, W < 32). */
#define ISX_RESNET50_CONVS 53
typedef struct {
  const isx_bf16* w[ISX_RESNET50_CONVS];
  const float* bias[ISX_RESNET50_CONVS];
} isx_resnet50_weights;
int64_t isx_resnet50_workspace_bytes(int B, int H, int W);
int isx_resnet50_forward(const isx_resnet50_weights* weights, const float* x, int xc, int B, int H, int W, void* workspace,
                         float* feat_out, isx_stream stream);

/* ---- evaluation metrics of the drivers ------------------------------------------------------------------------------------
 * isx_seg_iou = utils.cal_IoUs (utils.py:163-194; iris_style_transfer_openeds2019.py:156, data_preprocessing.py:168): preds,
 * targets int64 [B,HW] label maps -> iou fp32 [B,num_class] = intersection / (union + eps) per image and class, miou fp32 [B] =
 * their mean; one pass over the two maps (the reference makes ~30).  counts: uint32 [B,num_class,2] scratch (zeroed here).
 * Bit-identical to the reference (exact counts, the same fp32 division); num_class <= 8.
 * isx_angular_distance = utils.angular_distance (utils.py:216-240): rows v1, v2 fp32 [n,d] -> acos(clamp(<v1,v2>)) and degrees. */
int isx_seg_iou(const int64_t* preds, const int64_t* targets, int B, int64_t HW, int num_class, float eps, uint32_t* counts,
                float* iou, float* miou, isx_stream stream);
/* isx_seg_iou for two label maps of the same dtype: seg_dtype 0 = int64 (= isx_seg_iou), 1 = uint8 [B,HW] (2 B per pixel
 * instead of 16; any alignment and HW).  The counts are exact either way, so the results are bit-identical to the int64 call
 * on the widened maps.  Any other seg_dtype is an error. */
int isx_seg_iou_typed(const void* preds, const void* targets, int seg_dtype, int B, int64_t HW, int num_class, float eps,
                      uint32_t* counts, float* iou, float* miou, isx_stream stream);
int isx_angular_distance(const float* v1, const float* v2, int n, int d, float* radian, float* degree, isx_stream stream);

/* ---- measurement hooks (bench.py) -------------------------------------------------------------
 * isx_launch_count: kernels launched by this library since load.  isx_prof_enable(1) brackets every launch
 * of the tensor-core conv (family 0), Gram (1), L-BFGS pass (2) and landmark bit-plane (3) kernels with CUDA events on the
 * launching stream; after a device sync isx_prof_collect fills out[3*family + {0,1,2}] = {launches, total ms,
 * total algorithmic work (FLOPs for 0/1, bytes for 2/3)}; n_out >= 12. */
unsigned long long isx_launch_count(void);
/* kernel-selection options (defaults in parentheses).  The first four choose among kernels for the same convolution;
 * the default 1 picks one from the shapes of the call, 0 sends the call to the generic kernel, 2 forces the kernel on every
 * applicable call (tests compare each kernel with the generic one this way):
 *   "c64" (1): resident-weight kernel for the 64 -> 64 layers;
 *   "halo2" (1): halo-patch pair kernel for the mid layers;
 *   "tail_n" (1): taps-in-N image-gradient tail (0 or 1);
 *   "sweep64" (1): tap-stacked sweep kernel for the 64 -> 64 layers (conv_sweep.cu; 1: the forward launches whose 128-pixel
 *     strips fit the image).
 * "smem_reserve_kb" (0): shared memory per SM the persistent conv CTAs leave free (<= 22), so that one TMEM-free streaming CTA
 * of another stream -- the L-BFGS history passes -- can be resident beside them.
 * Unknown names return non-zero. */
int isx_set_option(const char* name, int value);   /* on the calling thread's current context */
int isx_get_option(const char* name, int* value);
int isx_prof_enable(int on);
int isx_prof_collect(double* out, int n_out);

#ifdef __cplusplus
}
#endif
#endif /* ISX_H_ */
