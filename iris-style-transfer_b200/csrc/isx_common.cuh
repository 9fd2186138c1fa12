// Common device/host helpers for the isx (iris style transfer, sm_100a) library:
// error plumbing, mbarrier / TMA / tcgen05 PTX wrappers, UMMA descriptors.
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

// ------------------------------------------------------------------------------------------
// host-side error plumbing (C-ABI returns int status; text via isx_last_error())
// ------------------------------------------------------------------------------------------
void isx_set_error(const char* fmt, ...);

#define ISX_CHECK_CUDA(expr)                                                              \
  do {                                                                                    \
    cudaError_t _e = (expr);                                                              \
    if (_e != cudaSuccess) {                                                              \
      isx_set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(_e)); \
      return 1;                                                                           \
    }                                                                                     \
  } while (0)

#define ISX_REQUIRE(cond, ...)   \
  do {                           \
    if (!(cond)) {               \
      isx_set_error(__VA_ARGS__); \
      return 2;                  \
    }                            \
  } while (0)

// ------------------------------------------------------------------------------------------
// Per-handle library state (isx_create / isx_destroy / isx_make_current, include/isx.h): kernel-selection options, the
// launch counter, the CUDA-event profiler and the device's SM count.  There is NO process-global mutable state: every
// entry point works on the calling thread's CURRENT context -- the handle it bound with isx_make_current, or a private
// default context created on first use (device = the thread's current CUDA device).
// ------------------------------------------------------------------------------------------
struct IsxProfiler;
struct IsxContext {
  int device = 0;
  int num_sms = 148;                 // cudaDevAttrMultiProcessorCount of `device` (B200: 148)
  int opt_c64 = 1;                   // "c64": resident-weight kernel for the 64 -> 64 layers (0 never, 1 heuristic, 2 always)
  int opt_halo2 = 1;                 // "halo2": halo-patch pair kernel for the mid layers
  int opt_tail_n = 1;                // "tail_n": taps-in-N image-gradient tail
  int opt_smem_reserve_kb = 0;       // "smem_reserve_kb": shared memory the persistent conv CTAs leave free per SM
  int opt_sweep64 = 1;               // "sweep64": tap-stacked sweep kernel for the 64 -> 64 layers (0 never, 1 = default: launches
                                     // whose 128-pixel strips fit the image and give every SM work, 2 always)
  unsigned long long launches = 0;   // kernels launched through this context
  IsxProfiler* prof = nullptr;
};
IsxContext* isx_ctx();
inline int isx_num_sms() { return isx_ctx()->num_sms; }

// every kernel launch of the library goes through this: error check + launch counter (bench.py's gpu_launches)
#define ISX_LAUNCH_CHECK()               \
  do {                                   \
    ++isx_ctx()->launches;               \
    ISX_CHECK_CUDA(cudaGetLastError());  \
  } while (0)

// optional CUDA-event timing of one kernel family on the launching stream (bench.py roofline leg)
void isx_prof_begin(int family, double work, cudaStream_t s);
void isx_prof_end(int family, cudaStream_t s);
enum { ISX_PROF_CONV = 0, ISX_PROF_GRAM = 1, ISX_PROF_LBFGS = 2, ISX_PROF_PLANES = 3, ISX_PROF_FAMILIES = 4 };

// Encode a tiled bf16 tensor map (rank <= 5).  dims/strides innermost first; strides in BYTES
// for dims 1..rank-1 (dim 0 is contiguous).  swizzle128: CU_TENSOR_MAP_SWIZZLE_128B else NONE.
// elem_strides (NULL = all 1): traversal stride per dim -- a box then lands ceil(box[i] / elem_strides[i]) elements of
// dim i, those at start, start + s, start + 2s, ... (strided convolutions).
int isx_make_tmap_bf16(CUtensorMap* out, const void* base, int rank, const uint64_t* dims,
                       const uint64_t* strides_bytes, const uint32_t* box, bool swizzle128,
                       const uint32_t* elem_strides = nullptr);

#ifdef __CUDACC__
namespace isx {

// SM count of the current context's device (host-side grid sizing only; kernels read gridDim)
#define kNumSMs (isx_num_sms())

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ uint32_t lane_id() { return threadIdx.x & 31; }

__device__ __forceinline__ bool elect_one() {
  uint32_t pred = 0;
  asm volatile(
      "{\n\t.reg .pred P;\n\t.reg .b32 R;\n\t"
      "elect.sync R|P, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, P;\n\t}"
      : "=r"(pred));
  return pred != 0;
}

// ---------------- mbarrier ----------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred P;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 P, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, P;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// Bounded wait: a pipeline bug must fault, not hang the GPU box (a hang is a strike).
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if (++spins > (1u << 26)) {
      printf("isx: mbarrier wait timed out (block %d,%d thread %d)\n", blockIdx.x, blockIdx.y, threadIdx.x);
      __trap();
    }
  }
}

// Wait on two barriers whose try_waits are issued back to back (the second does not wait for the first's result):
// an mbarrier probe costs ~100+ cycles even when the phase has long completed, and the MMA-issuing thread of a
// persistent kernel pays it once per barrier per tile.
__device__ __forceinline__ void mbar_wait2(uint64_t* bar_a, uint32_t parity_a, uint64_t* bar_b, uint32_t parity_b) {
  bool a = mbar_try_wait(bar_a, parity_a);
  bool b = mbar_try_wait(bar_b, parity_b);
  if (!a) mbar_wait(bar_a, parity_a);
  if (!b) mbar_wait(bar_b, parity_b);
}

// ---------------- TMA ----------------
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* smem, const CUtensorMap* m, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(smem)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d(void* smem, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(smem_u32(smem)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
__device__ __forceinline__ void tma_load_4d(void* smem, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2,
                                            int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(smem_u32(smem)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2),
      "r"(c3)
      : "memory");
}
__device__ __forceinline__ void tma_store_4d(const CUtensorMap* m, const void* smem, int c0, int c1, int c2, int c3) {
  asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];" ::"l"(
                   reinterpret_cast<uint64_t>(m)),
               "r"(smem_u32(smem)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
               : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void tma_store_wait_read() {
  asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
template <int N>
__device__ __forceinline__ void tma_store_wait_all() {
  asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory");
}

// ---------------- tcgen05 / TMEM ----------------
template <int kCols>
__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)),
               "n"(kCols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
template <int kCols>
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(kCols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// D[tmem] (+)= A[smem] * B[smem], kind::f16 (bf16 in, fp32 accumulate), single CTA.
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Same MMA with the descriptors split into 32-bit halves.  The issuing thread is the bottleneck of small-N tiles
// (measured: a single thread sustains one tcgen05.mma per ~49 cycles at best, ~70-100 with the descriptor rebuilt from
// the address every time -- scratch/umma_probe.cu, profiles/r01_umma_issue_probe.txt), so hot loops build the
// descriptor ONCE and add (byte offset >> 4) to the low word: the 14-bit address field cannot carry out for any
// shared-memory address below 256 KB.
__device__ __forceinline__ void umma_bf16_lohi(uint32_t tmem_d, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo, uint32_t b_hi,
                                               uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\t"
      "mov.b64 da, {%1, %2};\n\tmov.b64 db, {%3, %4};\n\t"
      "setp.ne.b32 p, %6, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %5, p;\n\t}"
      ::"r"(tmem_d), "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Arrive on an mbarrier when all previously issued tcgen05.mma of this thread have completed.
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}
// 32 lanes x 32 columns of fp32: thread i of the warp gets row (lane base + i), 32 consecutive columns.
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
        "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
        "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_32x16(uint32_t taddr, uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// Shared-memory matrix descriptor (sm_100: version=1 at bits 46-47), SWIZZLE_128B (layout type 2).
//   K-major : rows of 128 B (64 bf16 of K), 8-row swizzle atoms, SBO = byte stride between 8-row groups.
//   MN-major: rows of 128 B (64 bf16 of M/N) indexed by K, 8-K-row atoms at SBO, 64-wide MN blocks at LBO.
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes,
                                                   uint32_t base_offset = 0) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>(base_offset & 7) << 49;  // swizzle phase of the first row when start is not 1024-B aligned
  d |= static_cast<uint64_t>((smem_addr & 0x3FFFF) >> 4);
  d |= static_cast<uint64_t>((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= static_cast<uint64_t>((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= 1ull << 46;  // descriptor version (Blackwell)
  d |= 2ull << 61;  // SWIZZLE_128B
  return d;
}
// Instruction descriptor for kind::f16: bf16 x bf16 -> fp32.
__host__ __device__ constexpr uint32_t umma_idesc_bf16(int M, int N, bool a_mn_major, bool b_mn_major) {
  return (1u << 4)                              // c_format = F32
         | (1u << 7)                            // a_format = BF16
         | (1u << 10)                           // b_format = BF16
         | ((a_mn_major ? 1u : 0u) << 15)       // a_major
         | ((b_mn_major ? 1u : 0u) << 16)       // b_major
         | (static_cast<uint32_t>(N >> 3) << 17)  // n_dim
         | (static_cast<uint32_t>(M >> 4) << 24); // m_dim
}

// ---------------- small math helpers ----------------
__device__ __forceinline__ uint32_t pack_bf16x2(float a, float b) {
  __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&h);
}
__device__ __forceinline__ float2 unpack_bf16x2(uint32_t u) {
  __nv_bfloat162 h = *reinterpret_cast<__nv_bfloat162*>(&u);
  return __bfloat1622float2(h);
}
// 2x2 max-pool of four chunks of eight post-ReLU bf16 values (window scan order (0,0),(0,1),(1,0),(1,1)): the maxima and, per
// element, the ROUTING CODE of the fused max-pool + ReLU backward -- 0..3 = position of the FIRST maximum (ATen's
// `val > maxval` rule), 4 = blocked (maximum <= 0: ReLU passes nothing).  One byte per element, in element order.
__device__ __forceinline__ void pool4_codes(const uint4 (&u)[4], uint4& m4, uint2& codes) {
  uint32_t cw[4];
  const __nv_bfloat162 zero2 = __floats2bfloat162_rn(0.f, 0.f);
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    __nv_bfloat162 m = reinterpret_cast<const __nv_bfloat162*>(&u[0])[e];
    uint32_t code = 0u;
#pragma unroll
    for (int k = 1; k < 4; ++k) {
      const __nv_bfloat162 a = reinterpret_cast<const __nv_bfloat162*>(&u[k])[e];
      const uint32_t gt = __hgt2_mask(a, m);  // 0xFFFF per half where a > m
      m = __hmax2(m, a);
      code = (code & ~gt) | (gt & (static_cast<uint32_t>(k) * 0x00010001u));
    }
    const uint32_t z = __hle2_mask(m, zero2);
    cw[e] = (code & ~z) | (z & 0x00040004u);
    reinterpret_cast<__nv_bfloat162*>(&m4)[e] = m;
  }
  codes.x = __byte_perm(cw[0], cw[1], 0x6420);
  codes.y = __byte_perm(cw[2], cw[3], 0x6420);
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

}  // namespace isx
#endif  // __CUDACC__
