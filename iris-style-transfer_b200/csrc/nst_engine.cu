// Host-side driver of one NST closure evaluation (pipelines.py:80-91): VGG-19 forward to the deepest
// tap, style/content losses, backward to the image -- a fixed sequence of libisx kernels on one
// stream (graph-capturable: no allocation, no host synchronisation).  Also the L-BFGS C-ABI glue.
#include <algorithm>
#include <vector>

#include "../../include/isx.h"
#include "isx_common.cuh"
#include "isx_internal.h"
#include "isx_kernels.h"
#include "lbfgs_state.h"

using namespace isx;
typedef __nv_bfloat16 bf16;

static inline cudaStream_t S(isx_stream s) { return reinterpret_cast<cudaStream_t>(s); }

// torchvision vgg19 cfg "E" (torchvision/models/vgg.py:94): channels per conv, pool after convs 1,3,7,11,15
static const int kCout[16] = {64, 64, 128, 128, 256, 256, 256, 256, 512, 512, 512, 512, 512, 512, 512, 512};
static const int kCin[16] = {3, 64, 64, 128, 128, 256, 256, 256, 256, 512, 512, 512, 512, 512, 512, 512};
static const int kLevel[16] = {0, 0, 1, 1, 2, 2, 2, 2, 3, 3, 3, 3, 4, 4, 4, 4};  // resolution level = #pools before
static inline bool pool_after(int i) { return i == 1 || i == 3 || i == 7 || i == 11 || i == 15; }
// Tap ids (isx_nst_config.style_conv / content_conv): 0..15 = ReLU output of that conv, 16..20 = output of pool 0..4
// (models/vgg/vgg.py:6-10 lets any layer of vgg19.features be tapped, pools included).
static const int kConvBefore[5] = {1, 3, 7, 11, 15};
static inline int pool_index(int conv) { return conv == 1 ? 0 : conv == 3 ? 1 : conv == 7 ? 2 : conv == 11 ? 3 : 4; }
static inline bool tap_is_pool(int id) { return id >= ISX_TAP_POOL0; }
static inline int tap_conv(int id) { return tap_is_pool(id) ? kConvBefore[id - ISX_TAP_POOL0] : id; }   // the conv that must have run
static inline int tap_level(int id) { return tap_is_pool(id) ? id - ISX_TAP_POOL0 + 1 : kLevel[id]; }
static inline int tap_C(int id) { return kCout[tap_conv(id)]; }

namespace {
struct Layout {
  int B, H[6], W[6];
  size_t act[16];     // byte offsets of ReLU outputs
  size_t pool[5];     // byte offsets of pool outputs
  size_t pidx[5];     // routing bytes of each pool's backward (one per pooled element, pool4_codes)
  size_t gradA, gradB, tapbuf;
  size_t cgrad[ISX_MAX_TAPS];
  size_t gram_ws, D[ISX_MAX_TAPS], sums, csum, aff_a[ISX_MAX_TAPS], aff_b[ISX_MAX_TAPS];
  size_t fm2[ISX_MAX_TAPS], kbflags[ISX_MAX_TAPS];  // row G': F * m^2 (Gram-backward operand), non-zero K-block flags
  size_t total;
};

size_t align_up(size_t v) { return (v + 255) & ~size_t(255); }

int make_layout(const isx_nst_config* c, Layout* L) {
  ISX_REQUIRE(c->B > 0 && c->H > 0 && c->W > 0, "nst: empty batch");
  ISX_REQUIRE(c->n_conv >= 1 && c->n_conv <= 16, "nst: n_conv %d out of range", c->n_conv);
  ISX_REQUIRE(c->n_style >= 0 && c->n_style <= ISX_MAX_TAPS && c->n_content >= 0 && c->n_content <= ISX_MAX_TAPS,
              "nst: too many taps");
  L->B = c->B;
  L->H[0] = c->H; L->W[0] = c->W;
  for (int l = 1; l < 6; ++l) { L->H[l] = L->H[l - 1] / 2; L->W[l] = L->W[l - 1] / 2; }
  const int deepest_level = kLevel[c->n_conv - 1];
  ISX_REQUIRE(L->H[deepest_level] >= 1 && L->W[deepest_level] >= 1, "nst: image %dx%d too small for %d convs", c->H,
              c->W, c->n_conv);
  size_t off = 0;
  size_t max_act = 0, max_tap = 0;
  for (int i = 0; i < 16; ++i) {
    L->act[i] = off;
    if (i < c->n_conv) {
      const size_t bytes = static_cast<size_t>(c->B) * L->H[kLevel[i]] * L->W[kLevel[i]] * kCout[i] * 2;
      off += align_up(bytes);
      max_act = std::max(max_act, bytes);
    }
  }
  for (int k = 0; k < 5; ++k) {
    L->pool[k] = off;
    const int conv_before[5] = {1, 3, 7, 11, 15};
    if (conv_before[k] < c->n_conv)
      off += align_up(static_cast<size_t>(c->B) * L->H[k + 1] * L->W[k + 1] * kCout[conv_before[k]] * 2);
    L->pidx[k] = off;
    if (conv_before[k] < c->n_conv)
      off += align_up(static_cast<size_t>(c->B) * L->H[k + 1] * L->W[k + 1] * kCout[conv_before[k]]);
  }
  auto tap_ok = [&](int id) { return id >= 0 && id < ISX_VGG19_TAPS && tap_conv(id) < c->n_conv && L->H[tap_level(id)] >= 1 && L->W[tap_level(id)] >= 1; };
  for (int t = 0; t < c->n_style; ++t) {
    const int i = c->style_conv[t];
    ISX_REQUIRE(tap_ok(i), "nst: style tap conv %d beyond n_conv %d", i, c->n_conv);
    max_tap = std::max(max_tap, static_cast<size_t>(c->B) * L->H[tap_level(i)] * L->W[tap_level(i)] * tap_C(i) * 2);
  }
  L->gradA = off; off += align_up(max_act);
  L->gradB = off; off += align_up(max_act);
  L->tapbuf = off; off += align_up(std::max<size_t>(max_tap, 256));
  for (int t = 0; t < c->n_content; ++t) {
    const int i = c->content_conv[t];
    ISX_REQUIRE(tap_ok(i), "nst: content tap conv %d beyond n_conv %d", i, c->n_conv);
    L->cgrad[t] = off;
    off += align_up(static_cast<size_t>(c->B) * L->H[tap_level(i)] * L->W[tap_level(i)] * tap_C(i) * 2);
  }
  size_t gram_ws = 256, csum_ws = 256;
  for (int t = 0; t < c->n_style; ++t) {
    const int i = c->style_conv[t];
    const int C = tap_C(i);
    const int HW = L->H[tap_level(i)] * L->W[tap_level(i)];
    gram_ws = std::max<size_t>(gram_ws, static_cast<size_t>(gram_pick_splits(c->B, HW, C)) * c->B * C * C * 4);
    if (C <= 128) csum_ws = std::max<size_t>(csum_ws, static_cast<size_t>(gram_pick_splits(c->B, HW, C)) * c->B * C * 4);
    L->D[t] = off; off += align_up(static_cast<size_t>(c->B) * C * C * 2);
    L->aff_a[t] = off; off += align_up(static_cast<size_t>(c->B) * C * 4);
    L->aff_b[t] = off; off += align_up(static_cast<size_t>(c->B) * C * 4);
    L->fm2[t] = L->kbflags[t] = 0;
    if (c->style_mask_b > 0) {
      const size_t act_bytes = static_cast<size_t>(c->B) * HW * C * 2;
      L->fm2[t] = off; off += align_up(act_bytes);
      L->kbflags[t] = off; off += align_up(static_cast<size_t>(gram_mask_flags_bytes(c->style_mask_b, HW, C)));
    }
  }
  L->gram_ws = off; off += align_up(gram_ws);
  L->sums = off; off += align_up(static_cast<size_t>(c->B) * 512 * 2 * 8);
  L->csum = off; off += align_up(csum_ws);   // fused channel sums of the Gram kernel (feature extraction, C <= 128)
  L->total = off;
  return 0;
}

inline bf16* at(const isx_nst_buffers* b, size_t off) { return reinterpret_cast<bf16*>(static_cast<char*>(b->workspace) + off); }
inline float* atf(const isx_nst_buffers* b, size_t off) { return reinterpret_cast<float*>(static_cast<char*>(b->workspace) + off); }

inline size_t tap_off(const Layout& L, int id) { return tap_is_pool(id) ? L.pool[id - ISX_TAP_POOL0] : L.act[id]; }
bool pool_tapped(const isx_nst_config* c, int k) {
  for (int t = 0; t < c->n_style; ++t) if (c->style_conv[t] == ISX_TAP_POOL0 + k) return true;
  for (int t = 0; t < c->n_content; ++t) if (c->content_conv[t] == ISX_TAP_POOL0 + k) return true;
  return false;
}
int style_tap_of(const isx_nst_config* c, int conv) {
  for (int t = 0; t < c->n_style; ++t) if (c->style_conv[t] == conv) return t;
  return -1;
}
int content_tap_of(const isx_nst_config* c, int conv) {
  for (int t = 0; t < c->n_content; ++t) if (c->content_conv[t] == conv) return t;
  return -1;
}

inline uint8_t* atb(const isx_nst_buffers* b, size_t off) { return reinterpret_cast<uint8_t*>(static_cast<char*>(b->workspace) + off); }

// Is the ReLU output of conv `i` read by anything but the pool that follows it?  (taps only: the max-pool + ReLU backward
// routes through the pool's index bytes, not through the pre-pool activation)
bool conv_tapped(const isx_nst_config* c, int i) { return style_tap_of(c, i) >= 0 || content_tap_of(c, i) >= 0; }

// forward through conv `i` (input selection included).  lean: a pre-pool activation that no tap reads is not written to
// memory at all -- only its pooled map and the routing bytes are (57 MB of stores per 640x400 image).
int run_conv_fwd(const isx_nst_config* c, const isx_nst_buffers* b, const Layout& L, int i, const float* x,
                 bool want_pool, cudaStream_t s, bool lean = false) {
  const int lv = kLevel[i];
  if (i == 0 && b->w0_fwd != nullptr)
    return conv1_1_fwd_tc(x, c->xc, c->mask_b ? b->input_mask : nullptr, c->mask_b,
                          reinterpret_cast<const bf16*>(b->w0_fwd), b->bias[0], at(b, L.act[0]), c->B, L.H[0], L.W[0], s);
  if (i == 0)
    return conv1_1_fwd(x, c->xc, c->mask_b ? b->input_mask : nullptr, c->mask_b, b->w0, b->bias[0], at(b, L.act[0]), c->B,
                       L.H[0], L.W[0], s);
  const bool first_of_block = (i == 2 || i == 4 || i == 8 || i == 12);
  const bf16* in = first_of_block ? at(b, L.pool[lv - 1]) : at(b, L.act[i - 1]);
  ISX_REQUIRE(b->w_fwd[i] != nullptr, "nst: packed forward weights of conv %d missing", i);
  ConvArgs a;
  a.in = in; a.weight = reinterpret_cast<const bf16*>(b->w_fwd[i]); a.out = at(b, L.act[i]);
  a.B = c->B; a.H = L.H[lv]; a.W = L.W[lv]; a.Cin = kCin[i]; a.Cout = kCout[i]; a.ntaps = 9;
  a.bias = b->bias[i]; a.relu = 1;
  if (want_pool) {  // MaxPool2d(2,2) of this layer's output rides the conv epilogue
    ISX_REQUIRE(L.H[lv] >= 2 && L.W[lv] >= 2, "nst: cannot pool a %dx%d map", L.H[lv], L.W[lv]);
    a.pool_out = at(b, L.pool[lv]);
    a.pool_idx = atb(b, L.pidx[lv]);
    a.skip_out = lean && !conv_tapped(c, i);
  }
  return conv_tc(a, s);
}
}  // namespace

extern "C" int64_t isx_nst_workspace_bytes(const isx_nst_config* cfg) {
  Layout L;
  if (!cfg || make_layout(cfg, &L)) return -1;
  return static_cast<int64_t>(L.total);
}

extern "C" int isx_nst_forward(const isx_nst_config* c, const isx_nst_buffers* b, const float* x, int flags,
                               isx_stream stream) {
  ISX_REQUIRE(c && b && x && b->workspace, "isx_nst_forward: null pointer");
  Layout L;
  if (int rc = make_layout(c, &L)) return rc;
  cudaStream_t s = S(stream);
  const bool with_last_pool = (flags & ISX_FWD_LAST_POOL) != 0, lean = (flags & ISX_FWD_LEAN) != 0;
  for (int i = 0; i < c->n_conv; ++i) {
    const bool want_pool = pool_after(i) && (i + 1 < c->n_conv || with_last_pool || pool_tapped(c, pool_index(i)));
    if (int rc = run_conv_fwd(c, b, L, i, x, want_pool && i > 0, s, lean)) return rc;
    if (want_pool && i == 0) {  // (conv1_1 is never followed by a pool in VGG-19; kept for completeness)
      const int lv = kLevel[i];
      if (int rc = maxpool_fwd(at(b, L.act[i]), at(b, L.pool[lv]), c->B, L.H[lv], L.W[lv], kCout[i], s)) return rc;
    }
  }
  return 0;
}

extern "C" int isx_nst_feature(const isx_nst_config* c, const isx_nst_buffers* b, int kind, int idx, isx_bf16** ptr,
                               int32_t* h, int32_t* w, int32_t* ch) {
  ISX_REQUIRE(c && b && ptr && h && w && ch, "isx_nst_feature: null pointer");
  Layout L;
  if (int rc = make_layout(c, &L)) return rc;
  if (kind == 0) {
    ISX_REQUIRE(idx >= 0 && idx < c->n_conv, "isx_nst_feature: conv %d not computed (n_conv=%d)", idx, c->n_conv);
    *ptr = reinterpret_cast<isx_bf16*>(at(b, L.act[idx]));
    *h = L.H[kLevel[idx]]; *w = L.W[kLevel[idx]]; *ch = kCout[idx];
  } else {
    const int conv_before[5] = {1, 3, 7, 11, 15};
    ISX_REQUIRE(idx >= 0 && idx < 5 && conv_before[idx] < c->n_conv, "isx_nst_feature: pool %d not computed", idx);
    *ptr = reinterpret_cast<isx_bf16*>(at(b, L.pool[idx]));
    *h = L.H[idx + 1]; *w = L.W[idx + 1]; *ch = kCout[conv_before[idx]];
  }
  return 0;
}

namespace {
// Gradient sources arriving at the ReLU output of a conv (all optional): a ready bf16 gradient map, the per-channel
// affine form of the BN-statistics loss, and the Gram term D_b applied to gram_A (the activation or its masked copy).
struct TapSrc {
  const bf16* add = nullptr;
  const float* aa = nullptr;
  const float* ab = nullptr;
  const bf16* gram_D = nullptr;
  const bf16* gram_A = nullptr;
  bool add_is_masked = false;  // `add` is already multiplied by relu'(act) (content_mse output)
  bool any() const { return add || aa || gram_D; }
};

// Backward of the stored forward pass to the image: conv dgrad (tcgen05) chained through ReLU / max-pool backward with
// the tap gradients injected where they arise.  gm = ReLU-masked gradient w.r.t. a conv's output, ready for its dgrad.
int run_backward(const isx_nst_config* c, const isx_nst_buffers* b, const Layout& L, const TapSrc* src,
                 const bf16* last_pool_grad, float* grad, cudaStream_t s) {
  // src: ISX_VGG19_TAPS entries, [0..15] sources at conv ReLU outputs, [16..20] sources at pool outputs
  const int B = c->B;
  auto pool_src = [&](int conv) -> const TapSrc* {   // sources at the pool right after `conv`, if any
    if (!pool_after(conv)) return nullptr;
    const TapSrc& ps = src[ISX_TAP_POOL0 + pool_index(conv)];
    return ps.any() ? &ps : nullptr;
  };
  int deepest = c->n_conv - 1;  // start at the deepest conv that receives a gradient (layers above it contribute nothing)
  if (!last_pool_grad)
    while (deepest > 0 && !src[deepest].any() && !pool_src(deepest)) --deepest;
  bf16* ping = at(b, L.gradA);
  bf16* pong = at(b, L.gradB);
  bf16* tapbuf = at(b, L.tapbuf);
  const bf16* gm = nullptr;
  // out = A . D_b  [* relu'(A)]   (Gram tap gradient as a 1x1 tcgen05 GEMM with per-image weights); A lives at tap `id`
  auto gram_1x1 = [&](int id, bf16* out, bool mask) -> int {
    const int lv = tap_level(id);
    ConvArgs a;
    a.in = src[id].gram_A; a.weight = src[id].gram_D; a.out = out;
    a.B = B; a.H = L.H[lv]; a.W = L.W[lv]; a.Cin = tap_C(id); a.Cout = tap_C(id); a.ntaps = 1; a.per_image_weights = true;
    a.mask_act = mask ? at(b, tap_off(L, id)) : nullptr;
    return conv_tc(a, s);
  };
  // max-pool + ReLU backward of the pool after conv `conv` (level lv), through the routing bytes the forward left: the
  // pre-pool activation is not read (a lean forward never stores it)
  auto pool_bwd = [&](const bf16* dy, int lv, int conv, bf16* dx) -> int {
    return maxpool_bwd_idx(dy, atb(b, L.pidx[lv]), dx, B, L.H[lv], L.W[lv], kCout[conv], s);
  };
  // gradient w.r.t. a POOL output: out = g (may be NULL) + every source of that pool tap; no ReLU mask (the max-pool
  // backward that follows applies the ReLU mask of the pre-pool activation)
  auto pool_combine = [&](int k, const bf16* g, bf16* out) -> int {
    const int id = ISX_TAP_POOL0 + k, lv = k + 1, C = tap_C(id);
    const long HW = static_cast<long>(L.H[lv]) * L.W[lv];
    const TapSrc& t = src[id];
    const bf16* add2 = t.add;
    if (t.gram_D) {
      if (int rc = gram_1x1(id, tapbuf, false)) return rc;
      if (t.add)
        if (int rc = tap_add_mask(t.add, tapbuf, nullptr, nullptr, at(b, L.pool[k]), tapbuf, B, HW, C, s, 0)) return rc;
      add2 = tapbuf;
    }
    return tap_add_mask(g, add2, t.aa, t.ab, at(b, L.pool[k]), out, B, HW, C, s, 0);
  };
  {
    const int i = deepest, lv = kLevel[i], C = kCout[i];
    const long HW = static_cast<long>(L.H[lv]) * L.W[lv];
    const TapSrc& t = src[i];
    const bf16* up = nullptr;  // gradient arriving from above (only through the trailing pool)
    const bf16* pg = last_pool_grad;
    if (pool_src(i)) {          // taps on the pool after the deepest conv
      if (int rc = pool_combine(pool_index(i), pg, ping)) return rc;
      pg = ping;
    }
    if (pg) {
      if (int rc = pool_bwd(pg, lv, i, pong)) return rc;
      up = pong;
    }
    ISX_REQUIRE(up || t.any(), "nst backward: conv %d carries no gradient", i);
    if (up && !t.any()) {
      gm = up;  // the max-pool backward already applied this layer's ReLU mask (its activation may not even be stored)
    } else if (!up && t.add && !t.aa && !t.gram_D) {
      if (t.add_is_masked) {
        gm = t.add;
      } else {  // a lone gradient map must be ReLU-masked before the dgrad
        if (int rc = tap_add_mask(t.add, nullptr, nullptr, nullptr, at(b, L.act[i]), ping, B, HW, C, s)) return rc;
        gm = ping;
      }
    } else if (!up && !t.add && !t.aa && t.gram_D) {
      if (int rc = gram_1x1(i, ping, true)) return rc;
      gm = ping;
    } else {
      const bf16* add2 = nullptr;
      if (t.gram_D) {
        if (int rc = gram_1x1(i, tapbuf, false)) return rc;
        add2 = tapbuf;
      }
      // (up | add) + (gram | nothing) + affine, masked
      const bf16* g1 = up ? up : t.add;
      if (up && t.add && add2) {  // three maps: fold the given gradient into the tap buffer first
        if (int rc = tap_add_mask(t.add, tapbuf, nullptr, nullptr, at(b, L.act[i]), tapbuf, B, HW, C, s)) return rc;
      } else if (up && t.add) {
        add2 = t.add;
      }
      if (int rc = tap_add_mask(g1, add2, t.aa, t.ab, at(b, L.act[i]), ping, B, HW, C, s)) return rc;
      gm = ping;
    }
  }
  for (int i = deepest; i >= 1; --i) {
    const int lv = kLevel[i];
    const int j = i - 1;  // layer below
    const int lvj = kLevel[j];
    const int Cj = kCout[j];
    const long HWj = static_cast<long>(L.H[lvj]) * L.W[lvj];
    const TapSrc& t = src[j];
    const bool through_pool = pool_after(j);
    ConvArgs a;
    a.in = gm; a.weight = reinterpret_cast<const bf16*>(b->w_dgrad[i]);
    ISX_REQUIRE(b->w_dgrad[i] != nullptr, "nst: packed dgrad weights of conv %d missing", i);
    a.B = B; a.H = L.H[lv]; a.W = L.W[lv]; a.Cin = kCout[i]; a.Cout = kCin[i]; a.ntaps = 9;
    a.out = (gm == ping) ? pong : ping;
    bf16* other = (a.out == ping) ? pong : ping;
    if (!through_pool) {
      // tap gradients ride the dgrad: Gram term as extra K blocks of the main loop, map / affine terms in the epilogue
      a.mask_act = at(b, L.act[j]); a.add_buf = t.add; a.aff_a = t.aa; a.aff_b = t.ab;
      if (t.gram_D) { a.gram_act = t.gram_A; a.gram_D = t.gram_D; }
      if (int rc = conv_tc(a, s)) return rc;
      gm = a.out;
    } else {
      if (int rc = conv_tc(a, s)) return rc;  // gradient w.r.t. the pooled map: no ReLU
      if (pool_src(j))                        // taps on this pool add their gradient in place
        if (int rc = pool_combine(pool_index(j), a.out, a.out)) return rc;
      // `other` held this dgrad's input, which is consumed now
      if (int rc = pool_bwd(a.out, lvj, j, other)) return rc;
      gm = other;
      if (t.any()) {
        const bf16* add2 = t.add;
        if (t.gram_D) {
          if (int rc = gram_1x1(j, tapbuf, false)) return rc;
          if (t.add) {
            if (int rc = tap_add_mask(t.add, tapbuf, nullptr, nullptr, at(b, L.act[j]), tapbuf, B, HWj, Cj, s)) return rc;
          }
          add2 = tapbuf;
        }
        if (int rc = tap_add_mask(other, add2, t.aa, t.ab, at(b, L.act[j]), a.out, B, HWj, Cj, s)) return rc;
        gm = a.out;
      }
    }
  }
  if (b->w0_dgrad != nullptr) {
    ConvArgs a;
    a.in = gm; a.weight = reinterpret_cast<const bf16*>(b->w0_dgrad);
    a.B = B; a.H = L.H[0]; a.W = L.W[0]; a.Cin = 64; a.Cout = 16; a.ntaps = 9;
    a.dx_nchw = grad; a.xc = c->xc; a.in_mask = c->mask_b ? b->input_mask : nullptr; a.mask_b = c->mask_b;
    return conv_tc(a, s);
  }
  return conv1_1_dgrad(gm, b->w0, c->mask_b ? b->input_mask : nullptr, c->mask_b, grad, c->xc, B, L.H[0], L.W[0], s);
}
}  // namespace

namespace {
static_assert(kMaxRangedProblems == ISX_MAX_RANGED_PROBLEMS, "ProblemRanges holds the offsets of the largest layout");

// Several problems of one evaluation, validated by isx_nst_eval_problems / isx_nst_eval_ranges
struct ProblemSet {
  ProblemRanges r;
  int style_target_b;        // 1, P or B
  const double* c_weight;    // device [P]
  const double* s_weight;
};

// The checks isx_nst_eval_ranges and isx_lbfgs_tick_ranges share, before any device work: P within the limit, the offsets
// 0 = first_image[0] < ... < first_image[P] = B, the weight arrays; copies the offsets into r.
int load_ranges(const char* fn, const isx_nst_problem_ranges* pr, int B, ProblemRanges* r) {
  ISX_REQUIRE(pr && pr->first_image, "%s: null pointer", fn);
  const int P = pr->n_problems;
  ISX_REQUIRE(P >= 1 && P <= ISX_MAX_RANGED_PROBLEMS, "%s: problem count %d must be in 1..%d", fn, P, ISX_MAX_RANGED_PROBLEMS);
  ISX_REQUIRE(pr->first_image[0] == 0, "%s: first_image[0] = %d must be 0", fn, pr->first_image[0]);
  for (int p = 0; p < P; ++p)
    ISX_REQUIRE(pr->first_image[p + 1] > pr->first_image[p], "%s: first_image must increase strictly, problem %d is empty",
                fn, p);
  ISX_REQUIRE(pr->first_image[P] == B, "%s: first_image[%d] = %d must be the batch %d", fn, P, pr->first_image[P], B);
  ISX_REQUIRE(pr->c_weight && pr->s_weight, "%s: null per-problem weight array", fn);
  r->P = P;
  r->ipp = 0;
  for (int p = 0; p <= P; ++p) r->first[p] = pr->first_image[p];
  return 0;
}

// One closure evaluation.  ps == nullptr: the batch is one problem (c->coupled) or B problems, with the scalar weights of
// c.  Otherwise the batch is ps->r.P problems, each with its own alpha / beta (device arrays) and the style target of image
// b at 0, its problem or b (style target batch 1, P or B).
int nst_eval(const isx_nst_config* c, const isx_nst_buffers* b, const ProblemSet* ps, const float* x, double* loss_c,
             double* loss_s, float* grad, isx_stream stream) {
  Layout L;
  if (int rc = make_layout(c, &L)) return rc;
  cudaStream_t s = S(stream);
  const int B = c->B;
  const int deepest = c->n_conv - 1;
  const bool last_pool_tapped = pool_after(deepest) && pool_tapped(c, pool_index(deepest));
  ISX_REQUIRE(style_tap_of(c, deepest) >= 0 || content_tap_of(c, deepest) >= 0 || last_pool_tapped,
              "isx_nst_eval: conv %d is not tapped", deepest);
  ISX_CHECK_CUDA(cudaMemsetAsync(loss_c, 0, sizeof(double) * B, s));
  ISX_CHECK_CUDA(cudaMemsetAsync(loss_s, 0, sizeof(double) * B, s));
  // per-problem beta of the style taps: the finalize kernels form beta_p * w * k2 (Gram) or beta_p * w / k2 (BN)
  ProblemWeights pw;   // filled per tap below
  if (ps) {
    pw.r = ps->r;
    pw.target = ps->style_target_b == B ? 2 : ps->style_target_b == 1 ? 0 : 1;
  }
  auto style_weights = [&](double w, double k2) -> const ProblemWeights* {
    if (!ps) return nullptr;
    pw.weight = ps->s_weight; pw.k1 = w; pw.k2 = k2;
    return &pw;
  };

  // losses of everything tapped at `id` (a conv's ReLU output or a pool output), evaluated on the stored activation
  auto tap_losses = [&](int id) -> int {
    const int lv = tap_level(id);
    const int C = tap_C(id);
    const long HW = static_cast<long>(L.H[lv]) * L.W[lv];
    const bf16* act = at(b, tap_off(L, id));
    const int st = style_tap_of(c, id);
    if (st >= 0) {
      const double w = c->style_w[st];
      if (c->style_mode == 0) {  // StyleLoss_Gram (utils.py:317-322); GramMatrix n = C*H*W (utils.py:254)
        ISX_REQUIRE(b->gram_target[st], "nst: Gram target %d missing", st);
        const double inv_n = 1.0 / ((c->pred_unbatched ? 1.0 : static_cast<double>(C)) * HW);
        GramMask gm;
        if (c->style_mask_b > 0) {  // row G': Gram of F * m_l, weights applied to the operand tile inside the Gram kernel
          ISX_REQUIRE(b->style_mask[st], "nst: style mask %d missing", st);
          gm.m = b->style_mask[st]; gm.mask_b = c->style_mask_b;
          gm.kb_flags = reinterpret_cast<const uint8_t*>(at(b, L.kbflags[st]));  // isx_nst_prepare_style_masks
          gm.fm2 = at(b, L.fm2[st]);
        }
        const int splits = gram_pick_splits(B, static_cast<int>(HW), C);
        int rc = gram_sym_partial(act, B, static_cast<int>(HW), C, splits, atf(b, L.gram_ws), c->style_mask_b > 0 ? &gm : nullptr, s);
        if (rc) return rc;
        rc = gram_finalize(atf(b, L.gram_ws), B, splits, C, static_cast<float>(inv_n), nullptr, b->gram_target[st],
                           c->style_target_b, 0.25 * w, loss_s, static_cast<float>(c->s_weight * w * inv_n), at(b, L.D[st]), s,
                           nullptr, 0, style_weights(w, inv_n));
        if (rc) return rc;
      } else {  // StyleLoss_BN (utils.py:350-355)
        ISX_REQUIRE(b->bn_target_mean[st] && b->bn_target_std[st], "nst: BN target %d missing", st);
        ISX_REQUIRE(HW >= 2, "nst: unbiased std needs >= 2 pixels at tap %d", id);
        double* sums = reinterpret_cast<double*>(static_cast<char*>(b->workspace) + L.sums);
        ISX_CHECK_CUDA(cudaMemsetAsync(sums, 0, sizeof(double) * B * C * 2, s));
        const float* m = nullptr;
        if (c->style_mask_b > 0) {  // mask-weighted variant: StyleLoss_BN(F * m_l), statistics of the weighted features
          ISX_REQUIRE(b->style_mask[st], "nst: style mask %d missing", st);
          m = b->style_mask[st];
        }
        int rc = chan_sums(act, B, HW, C, sums, s, m, c->style_mask_b);
        if (rc) return rc;
        rc = bn_finalize(sums, B, C, HW, nullptr, nullptr, b->bn_target_mean[st], b->bn_target_std[st],
                         c->style_target_b, w / C, c->s_weight * w / C, loss_s, atf(b, L.aff_a[st]), atf(b, L.aff_b[st]), s,
                         0, style_weights(w, static_cast<double>(C)));
        if (rc) return rc;
        if (m)  // the gradient is no longer affine in F alone: m a + m^2 b F, materialised as a gradient map (buffer fm2)
          if (int rc2 = masked_affine_grad(act, m, c->style_mask_b, atf(b, L.aff_a[st]), atf(b, L.aff_b[st]), at(b, L.fm2[st]), B, HW, C, s)) return rc2;
      }
    }
    const int ct = content_tap_of(c, id);
    if (ct >= 0) {  // ContentLoss_L2 (utils.py:285-290): 0.5 * w * mean((p-t)^2)
      ISX_REQUIRE(b->content_target[ct], "nst: content target %d missing", ct);
      const long per_image = HW * C;
      // F.mse_loss over the problem's batch: B images when coupled, else one; with several problems the kernel forms
      // per_image * g_p itself
      const double denom = static_cast<double>(per_image) * (c->coupled ? B : 1);
      if (ps) { pw.weight = ps->c_weight; pw.k1 = c->content_w[ct]; pw.k2 = static_cast<double>(per_image); }
      int rc = content_mse(act, reinterpret_cast<const bf16*>(b->content_target[ct]), c->content_target_b,
                           at(b, L.cgrad[ct]), B, per_image, 0.5 * c->content_w[ct] / denom,
                           static_cast<float>(c->c_weight * c->content_w[ct] / denom), loss_c, s, 1, ps ? &pw : nullptr);
      if (rc) return rc;
    }
    return 0;
  };

  // ---------------- forward + losses ----------------
  for (int i = 0; i < c->n_conv; ++i) {
    const bool want_pool = pool_after(i) && (i + 1 < c->n_conv || pool_tapped(c, pool_index(i)));
    if (int rc = run_conv_fwd(c, b, L, i, x, want_pool, s, /*lean=*/true)) return rc;
    if (int rc = tap_losses(i)) return rc;
    if (want_pool && pool_tapped(c, pool_index(i)))
      if (int rc = tap_losses(ISX_TAP_POOL0 + pool_index(i))) return rc;
  }

  // ---------------- backward ----------------
  TapSrc src[ISX_VGG19_TAPS];
  for (int id = 0; id < ISX_VGG19_TAPS; ++id) {
    if (tap_conv(id) >= c->n_conv) continue;
    const int st = style_tap_of(c, id), ct = content_tap_of(c, id);
    if (ct >= 0) { src[id].add = at(b, L.cgrad[ct]); src[id].add_is_masked = true; }  // content_mse masks its gradient
    if (st >= 0 && c->style_mode == 0) {
      src[id].gram_D = at(b, L.D[st]);
      src[id].gram_A = c->style_mask_b > 0 ? at(b, L.fm2[st]) : at(b, tap_off(L, id));
    } else if (st >= 0 && c->style_mask_b > 0) {   // masked BN loss: a ready gradient map
      if (src[id].add) {  // a content tap on the same layer already supplies a map: sum them
        const long HWt = static_cast<long>(L.H[tap_level(id)]) * L.W[tap_level(id)];
        if (int rc = tap_add_mask(src[id].add, at(b, L.fm2[st]), nullptr, nullptr, at(b, tap_off(L, id)), at(b, L.fm2[st]), B, HWt,
                                  tap_C(id), s, 0)) return rc;
      }
      src[id].add = at(b, L.fm2[st]);
      src[id].add_is_masked = false;
    } else if (st >= 0) {
      src[id].aa = atf(b, L.aff_a[st]);
      src[id].ab = atf(b, L.aff_b[st]);
    }
  }
  return run_backward(c, b, L, src, nullptr, grad, s);
}
}  // namespace

extern "C" int isx_nst_eval(const isx_nst_config* c, const isx_nst_buffers* b, const float* x, double* loss_c,
                            double* loss_s, float* grad, isx_stream stream) {
  ISX_REQUIRE(c && b && x && loss_c && loss_s && grad && b->workspace, "isx_nst_eval: null pointer");
  ISX_REQUIRE(c->n_style + c->n_content > 0, "isx_nst_eval: no loss taps");
  ISX_REQUIRE(c->style_mask_b == 0 || c->style_mask_b == 1 || c->style_mask_b == c->B, "isx_nst_eval: style mask batch %d", c->style_mask_b);
  return nst_eval(c, b, nullptr, x, loss_c, loss_s, grad, stream);
}

extern "C" int isx_nst_eval_problems(const isx_nst_config* c, const isx_nst_buffers* b, const isx_nst_problems* pr,
                                     const float* x, double* loss_c, double* loss_s, float* grad, isx_stream stream) {
  ISX_REQUIRE(c && b && pr && x && loss_c && loss_s && grad && b->workspace, "isx_nst_eval_problems: null pointer");
  ISX_REQUIRE(c->n_style + c->n_content > 0, "isx_nst_eval_problems: no loss taps");
  const int B = c->B, g = pr->images_per_problem;
  ISX_REQUIRE(B > 0 && g >= 1 && B % g == 0, "isx_nst_eval_problems: batch %d is not a whole number of problems of %d images",
              B, g);
  const int P = B / g, tb = pr->style_target_b;
  ISX_REQUIRE(c->n_style == 0 || tb == 1 || tb == P || tb == B,
              "isx_nst_eval_problems: style target batch %d must be 1, %d (problems) or %d (images)", tb, P, B);
  ISX_REQUIRE(pr->c_weight && pr->s_weight, "isx_nst_eval_problems: null per-problem weight array");
  ISX_REQUIRE(c->style_mask_b == 0 || c->style_mask_b == 1 || c->style_mask_b == B,
              "isx_nst_eval_problems: style mask batch %d", c->style_mask_b);
  ProblemSet ps;
  ps.r.P = P;
  ps.r.ipp = g;
  ps.style_target_b = c->n_style == 0 ? B : tb;   // no target is read without style taps
  ps.c_weight = pr->c_weight;
  ps.s_weight = pr->s_weight;
  return nst_eval(c, b, &ps, x, loss_c, loss_s, grad, stream);
}

extern "C" int isx_nst_eval_ranges(const isx_nst_config* c, const isx_nst_buffers* b, const isx_nst_problem_ranges* pr,
                                   const float* x, double* loss_c, double* loss_s, float* grad, isx_stream stream) {
  ISX_REQUIRE(c && b && pr && x && loss_c && loss_s && grad && b->workspace, "isx_nst_eval_ranges: null pointer");
  ISX_REQUIRE(c->n_style + c->n_content > 0, "isx_nst_eval_ranges: no loss taps");
  const int B = c->B;
  ProblemSet ps;
  if (int rc = load_ranges("isx_nst_eval_ranges", pr, B, &ps.r)) return rc;
  const int P = ps.r.P, tb = pr->style_target_b;
  ISX_REQUIRE(c->n_style == 0 || tb == 1 || tb == P || tb == B,
              "isx_nst_eval_ranges: style target batch %d must be 1, %d (problems) or %d (images)", tb, P, B);
  ISX_REQUIRE(c->style_mask_b == 0 || c->style_mask_b == 1 || c->style_mask_b == B,
              "isx_nst_eval_ranges: style mask batch %d", c->style_mask_b);
  ps.style_target_b = c->n_style == 0 ? B : tb;
  ps.c_weight = pr->c_weight;
  ps.s_weight = pr->s_weight;
  return nst_eval(c, b, &ps, x, loss_c, loss_s, grad, stream);
}

extern "C" int isx_nst_prepare_style_masks(const isx_nst_config* c, const isx_nst_buffers* b, isx_stream stream) {
  ISX_REQUIRE(c && b && b->workspace, "isx_nst_prepare_style_masks: null pointer");
  ISX_REQUIRE(c->style_mask_b == 1 || c->style_mask_b == c->B, "isx_nst_prepare_style_masks: style mask batch %d", c->style_mask_b);
  Layout L;
  if (int rc = make_layout(c, &L)) return rc;
  cudaStream_t s = S(stream);
  if (c->style_mode != 0) return 0;  // mask-weighted BN loss: the mask is read directly by the statistics / gradient kernels
  for (int t = 0; t < c->n_style; ++t) {
    const int i = c->style_conv[t];
    const int C = tap_C(i);
    const int HW = L.H[tap_level(i)] * L.W[tap_level(i)];
    ISX_REQUIRE(b->style_mask[t], "isx_nst_prepare_style_masks: style mask %d missing", t);
    // F * m^2 is rewritten by every evaluation on the K blocks whose mask is not all zero; everything else stays zero
    ISX_CHECK_CUDA(cudaMemsetAsync(at(b, L.fm2[t]), 0, static_cast<size_t>(c->B) * HW * C * 2, s));
    if (int rc = gram_mask_flags(b->style_mask[t], c->style_mask_b, HW, C, reinterpret_cast<uint8_t*>(at(b, L.kbflags[t])), s))
      return rc;
  }
  return 0;
}

// Style features of the batch the preceding isx_nst_forward left in the workspace (classifiers.py:71 statistics and
// the utils.GramMatrix upper triangles), written straight into the caller's row-major matrix.
extern "C" int isx_nst_style_features(const isx_nst_config* c, const isx_nst_buffers* b, int want_stats, int want_gram,
                                      float* out, int64_t ld, isx_stream stream) {
  ISX_REQUIRE(c && b && out && b->workspace, "isx_nst_style_features: null pointer");
  ISX_REQUIRE(want_stats || want_gram, "isx_nst_style_features: nothing to extract");
  Layout L;
  if (int rc = make_layout(c, &L)) return rc;
  cudaStream_t s = S(stream);
  const int B = c->B;
  int64_t need = 0;
  for (int t = 0; t < c->n_style; ++t) {
    const int64_t C = tap_C(c->style_conv[t]);
    need += (want_stats ? 2 * C : 0) + (want_gram ? C * (C + 1) / 2 : 0);
  }
  ISX_REQUIRE(ld >= need, "isx_nst_style_features: row stride %lld < feature dimension %lld", (long long)ld, (long long)need);
  // column offsets: [per tap: mean | std] then [per tap: Gram upper triangle]
  int64_t stat_off[ISX_MAX_TAPS], gram_off[ISX_MAX_TAPS], off = 0;
  for (int t = 0; t < c->n_style; ++t) { stat_off[t] = off; if (want_stats) off += 2 * tap_C(c->style_conv[t]); }
  for (int t = 0; t < c->n_style; ++t) { gram_off[t] = off; if (want_gram) off += static_cast<int64_t>(tap_C(c->style_conv[t])) * (tap_C(c->style_conv[t]) + 1) / 2; }
  double* sums = reinterpret_cast<double*>(static_cast<char*>(b->workspace) + L.sums);
  for (int t = 0; t < c->n_style; ++t) {
    const int i = c->style_conv[t], lv = tap_level(i), C = tap_C(i);
    const int HW = L.H[lv] * L.W[lv];
    ISX_REQUIRE(!want_stats || HW >= 2, "isx_nst_style_features: unbiased std needs >= 2 pixels at conv %d", i);
    const int splits = gram_pick_splits(B, HW, C);
    // C <= 128 (HBM-bound layers, 80 % of the feature bytes): when both outputs are wanted, the statistics come out of the
    // Gram pass itself -- sum f from one extra N = 16 MMA per 16 pixels, sum f^2 from the Gram diagonal -- instead of a
    // second pass over the map
    const bool fused = want_stats && want_gram && C <= 128;
    if (want_stats && !fused) {
      ISX_CHECK_CUDA(cudaMemsetAsync(sums, 0, sizeof(double) * B * C * 2, s));
      if (int rc = chan_sums(at(b, tap_off(L, i)), B, HW, C, sums, s)) return rc;
      if (int rc = bn_finalize(sums, B, C, HW, out + stat_off[t], out + stat_off[t] + C, nullptr, nullptr, 1, 0.0, 0.0, nullptr,
                               nullptr, nullptr, s, ld)) return rc;
    }
    if (want_gram) {
      float* csum = fused ? atf(b, L.csum) : nullptr;
      if (int rc = gram_sym_partial(at(b, tap_off(L, i)), B, HW, C, splits, atf(b, L.gram_ws), nullptr, s, csum)) return rc;
      if (fused)
        if (int rc = stats_from_gram(atf(b, L.gram_ws), csum, B, splits, C, HW, out + stat_off[t], out + stat_off[t] + C, ld, s)) return rc;
      if (int rc = gram_finalize(atf(b, L.gram_ws), B, splits, C, static_cast<float>(1.0 / (static_cast<double>(C) * HW)),
                                 nullptr, nullptr, 1, 0.0, nullptr, 0.f, nullptr, s, out + gram_off[t], ld)) return rc;
    }
  }
  return 0;
}

extern "C" int isx_nst_backward(const isx_nst_config* c, const isx_nst_buffers* b, const isx_bf16* const* feat_grads,
                                const isx_bf16* last_pool_grad, float* grad, isx_stream stream) {
  ISX_REQUIRE(c && b && feat_grads && grad && b->workspace, "isx_nst_backward: null pointer");
  Layout L;
  if (int rc = make_layout(c, &L)) return rc;
  TapSrc src[ISX_VGG19_TAPS];
  bool any = last_pool_grad != nullptr;
  for (int id = 0; id < ISX_VGG19_TAPS; ++id) {
    if (tap_conv(id) >= c->n_conv) continue;
    src[id].add = reinterpret_cast<const bf16*>(feat_grads[id]);
    any = any || src[id].add != nullptr;
  }
  ISX_REQUIRE(any, "isx_nst_backward: no gradient given");
  ISX_REQUIRE(!last_pool_grad || pool_after(c->n_conv - 1), "isx_nst_backward: conv %d is not followed by a pool", c->n_conv - 1);
  return run_backward(c, b, L, src, reinterpret_cast<const bf16*>(last_pool_grad), grad, S(stream));
}

// ---------------------------------------------------------------------------------------------
// L-BFGS C-ABI glue
// ---------------------------------------------------------------------------------------------
extern "C" int64_t isx_lbfgs_state_bytes(int P) { return static_cast<int64_t>(P) * sizeof(LbfgsState); }
extern "C" int64_t isx_lbfgs_mats_bytes(int P, int history) {
  return static_cast<int64_t>(P) * 3 * (history + 1) * (history + 1) * 8;
}
extern "C" int64_t isx_lbfgs_scratch_bytes(int P, int64_t N, int history) {
  const int64_t nblk = lbfgs_nblk(N);
  const int64_t floats = P * nblk * (static_cast<int64_t>(history + 1) * 4 + 4);
  return ((floats * 4 + 255) / 256) * 256 + static_cast<int64_t>(P) * (history + 2) * 4 * 8 + 256;
}
extern "C" int isx_lbfgs_init(void* state, int P, isx_stream stream) {
  ISX_REQUIRE(state && P > 0, "isx_lbfgs_init: bad arguments");
  return lbfgs_init(static_cast<LbfgsState*>(state), P, S(stream));
}
namespace {
int lbfgs_tick_impl(float* x, const float* grad, float* grad_prev, void* Sh, void* Yh, void* state, void* mats, void* scratch,
                    const double* loss_c, const double* loss_s, int images_per_problem, int P, int64_t N,
                    const isx_lbfgs_config* cfg, const double* c_weight, const double* s_weight, double* hist_c,
                    double* hist_s, int tick, isx_stream stream, const ProblemRanges* pr = nullptr) {
  LbfgsConfig lc;
  lc.epochs = cfg->epochs; lc.max_iter = cfg->max_iter; lc.max_eval = cfg->max_eval; lc.history = cfg->history;
  lc.lr = cfg->lr; lc.tolerance_grad = cfg->tolerance_grad; lc.tolerance_change = cfg->tolerance_change;
  lc.c_weight = cfg->c_weight; lc.s_weight = cfg->s_weight;
  const int nblk = lbfgs_nblk(N);
  float* part = static_cast<float*>(scratch);
  float* ext = part + static_cast<int64_t>(P) * nblk * (cfg->history + 1) * 4;
  const int64_t floats = static_cast<int64_t>(P) * nblk * (static_cast<int64_t>(cfg->history + 1) * 4 + 4);
  double* dots = reinterpret_cast<double*>(static_cast<char*>(scratch) + ((floats * 4 + 255) / 256) * 256);
  return lbfgs_tick(x, grad, grad_prev, Sh, Yh, cfg->history_bf16, static_cast<LbfgsState*>(state), static_cast<double*>(mats), part, ext,
                    dots, loss_c, loss_s, images_per_problem, P, N, lc, hist_c, hist_s, tick, S(stream), c_weight, s_weight, pr);
}
}  // namespace

extern "C" int isx_lbfgs_tick(float* x, const float* grad, float* grad_prev, void* Sh, void* Yh, void* state,
                              void* mats, void* scratch, const double* loss_c, const double* loss_s,
                              int images_per_problem, int P, int64_t N, const isx_lbfgs_config* cfg, double* hist_c,
                              double* hist_s, int tick, isx_stream stream) {
  ISX_REQUIRE(x && grad && grad_prev && Sh && Yh && state && mats && scratch && loss_c && loss_s && cfg && hist_c && hist_s,
              "isx_lbfgs_tick: null pointer");
  ISX_REQUIRE(cfg->history >= 1 && cfg->history <= 100, "isx_lbfgs_tick: history %d must be in 1..100", cfg->history);
  return lbfgs_tick_impl(x, grad, grad_prev, Sh, Yh, state, mats, scratch, loss_c, loss_s, images_per_problem, P, N, cfg,
                         nullptr, nullptr, hist_c, hist_s, tick, stream);
}

extern "C" int isx_lbfgs_tick_problems(float* x, const float* grad, float* grad_prev, void* Sh, void* Yh, void* state,
                                       void* mats, void* scratch, const double* loss_c, const double* loss_s,
                                       int images_per_problem, int P, int64_t N, const isx_lbfgs_config* cfg,
                                       const double* c_weight, const double* s_weight, double* hist_c, double* hist_s,
                                       int tick, isx_stream stream) {
  ISX_REQUIRE(x && grad && grad_prev && Sh && Yh && state && mats && scratch && loss_c && loss_s && cfg && hist_c && hist_s,
              "isx_lbfgs_tick_problems: null pointer");
  ISX_REQUIRE(c_weight && s_weight, "isx_lbfgs_tick_problems: null per-problem weight array");
  ISX_REQUIRE(images_per_problem >= 1 && P >= 1 && N >= 1, "isx_lbfgs_tick_problems: %d problems of %d images, N = %lld",
              P, images_per_problem, (long long)N);
  ISX_REQUIRE(cfg->history >= 1 && cfg->history <= 100, "isx_lbfgs_tick_problems: history %d must be in 1..100",
              cfg->history);
  ProblemRanges r;
  r.P = P;
  r.ipp = images_per_problem;
  r.n = N;
  return lbfgs_tick_impl(x, grad, grad_prev, Sh, Yh, state, mats, scratch, loss_c, loss_s, images_per_problem, P, N, cfg,
                         c_weight, s_weight, hist_c, hist_s, tick, stream, &r);
}

extern "C" int isx_lbfgs_tick_ranges(float* x, const float* grad, float* grad_prev, void* Sh, void* Yh, void* state,
                                     void* mats, void* scratch, const double* loss_c, const double* loss_s,
                                     const isx_nst_problem_ranges* ranges, int B, int64_t n_img,
                                     const isx_lbfgs_config* cfg, double* hist_c, double* hist_s, int tick,
                                     isx_stream stream) {
  ISX_REQUIRE(x && grad && grad_prev && Sh && Yh && state && mats && scratch && loss_c && loss_s && cfg && hist_c && hist_s,
              "isx_lbfgs_tick_ranges: null pointer");
  ProblemRanges r;
  if (int rc = load_ranges("isx_lbfgs_tick_ranges", ranges, B, &r)) return rc;
  ISX_REQUIRE(n_img >= 1, "isx_lbfgs_tick_ranges: %lld elements per image", (long long)n_img);
  ISX_REQUIRE(cfg->history >= 1 && cfg->history <= 100, "isx_lbfgs_tick_ranges: history %d must be in 1..100", cfg->history);
  r.n = n_img;
  int g_max = 0;   // the grid of both history passes spans the largest problem
  for (int p = 0; p < r.P; ++p) g_max = std::max(g_max, r.size(p));
  return lbfgs_tick_impl(x, grad, grad_prev, Sh, Yh, state, mats, scratch, loss_c, loss_s, 0, r.P, g_max * n_img, cfg,
                         ranges->c_weight, ranges->s_weight, hist_c, hist_s, tick, stream, &r);
}

__global__ void done_flags_kernel(const LbfgsState* st, int P, int32_t* out) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p < P) out[p] = st[p].done ? st[p].func_evals : 0;
}
extern "C" int isx_lbfgs_done_flags(const void* state, int P, int32_t* done_out, isx_stream stream) {
  ISX_REQUIRE(state && done_out, "isx_lbfgs_done_flags: null pointer");
  done_flags_kernel<<<(P + 127) / 128, 128, 0, S(stream)>>>(static_cast<const LbfgsState*>(state), P, done_out);
  ISX_LAUNCH_CHECK();
  return 0;
}
__global__ void history_counts_kernel(const LbfgsState* st, int P, int32_t* out) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p < P) out[p] = st[p].hist_count;
}
extern "C" int isx_lbfgs_history_counts(const void* state, int P, int32_t* count_out, isx_stream stream) {
  ISX_REQUIRE(state && count_out, "isx_lbfgs_history_counts: null pointer");
  history_counts_kernel<<<(P + 127) / 128, 128, 0, S(stream)>>>(static_cast<const LbfgsState*>(state), P, count_out);
  ISX_LAUNCH_CHECK();
  return 0;
}
extern "C" int isx_clamp01(float* x, int64_t n, isx_stream stream) {
  ISX_REQUIRE(x && n >= 0, "isx_clamp01: bad arguments");
  return clamp01(x, n, S(stream));
}
