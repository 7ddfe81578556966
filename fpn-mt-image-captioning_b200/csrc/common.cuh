// Shared device/host helpers for the sm_100a kernels: error handling, activation views,
// bf16 packing, and thin inline-PTX wrappers for mbarrier / TMA / tcgen05 / TMEM.
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include <string>

namespace fpnmt {

typedef __nv_bfloat16 bf16;

// host bf16 conversion of weights: round-to-nearest-even, matches __float2bfloat16_rn for finite values
inline uint16_t f2bf(float f) {
  uint32_t u;
  memcpy(&u, &f, 4);
  if ((u & 0x7fffffffu) > 0x7f800000u) return 0x7fc0;
  u += 0x7fffu + ((u >> 16) & 1u);
  return (uint16_t)(u >> 16);
}
inline float bf2f(uint16_t h) {
  uint32_t u = (uint32_t)h << 16;
  float f;
  memcpy(&f, &u, 4);
  return f;
}

// ------------------------------------------------------------------------------------------------
// error plumbing (host)
// ------------------------------------------------------------------------------------------------
void set_last_error(const std::string& s);
#define FPNMT_CUDA_OK(expr)                                                                         \
  do {                                                                                              \
    cudaError_t _e = (expr);                                                                        \
    if (_e != cudaSuccess) {                                                                        \
      ::fpnmt::set_last_error(std::string(#expr) + " failed: " + cudaGetErrorString(_e) + " at " +   \
                              __FILE__ + ":" + std::to_string(__LINE__));                           \
      return 3; /* FPNMT_ERR_CUDA */                                                                \
    }                                                                                               \
  } while (0)

// ------------------------------------------------------------------------------------------------
// Activation view.  An activation tensor is [pixels][ld] bf16.  In the BF16X3 ("split") precision
// mode each value v is stored as hi = bf16(v) at [c] and lo = bf16(v - hi) at [lo + c]; lo == 0
// means plain bf16 storage.
// ------------------------------------------------------------------------------------------------
struct Act {
  bf16* p;
  int C;    // logical channels
  int ld;   // elements between consecutive pixels (rows)
  int lo;   // element offset of the low halves (0 = not split)
};

enum ActFn { ACT_NONE = 0, ACT_RELU = 1, ACT_LEAKY = 2, ACT_RELU6 = 3 };

__device__ __forceinline__ float apply_act(float v, int act) {
  if (act == ACT_RELU) return fmaxf(v, 0.f);
  if (act == ACT_LEAKY) return v >= 0.f ? v : 0.2f * v;
  if (act == ACT_RELU6) return fminf(fmaxf(v, 0.f), 6.f);
  return v;
}

__device__ __forceinline__ float ld_act(const Act& a, size_t pix, int c) {
  const bf16* q = a.p + pix * (size_t)a.ld + c;
  float v = __bfloat162float(q[0]);
  if (a.lo) v += __bfloat162float(q[a.lo]);
  return v;
}
__device__ __forceinline__ void st_act(const Act& a, size_t pix, int c, float v) {
  bf16* q = a.p + pix * (size_t)a.ld + c;
  bf16 h = __float2bfloat16_rn(v);
  q[0] = h;
  if (a.lo) q[a.lo] = __float2bfloat16_rn(v - __bfloat162float(h));
}

// 8-wide (16 byte) vector access; c must be a multiple of 8 and the view 16B aligned.
__device__ __forceinline__ void unpack8(const uint4& u, float* f) {
  const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    f[2 * i] = __uint_as_float(w[i] << 16);
    f[2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u);
  }
}
__device__ __forceinline__ uint32_t pack2(float a, float b) {
  __nv_bfloat162 t = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&t);
}
__device__ __forceinline__ uint4 pack8(const float* f) {
  return make_uint4(pack2(f[0], f[1]), pack2(f[2], f[3]), pack2(f[4], f[5]), pack2(f[6], f[7]));
}
__device__ __forceinline__ void ld_act8(const Act& a, size_t pix, int c, float* f) {
  const bf16* q = a.p + pix * (size_t)a.ld + c;
  unpack8(*reinterpret_cast<const uint4*>(q), f);
  if (a.lo) {
    float g[8];
    unpack8(*reinterpret_cast<const uint4*>(q + a.lo), g);
#pragma unroll
    for (int i = 0; i < 8; ++i) f[i] += g[i];
  }
}
__device__ __forceinline__ void st_act8(const Act& a, size_t pix, int c, const float* f) {
  bf16* q = a.p + pix * (size_t)a.ld + c;
  uint4 h = pack8(f);
  *reinterpret_cast<uint4*>(q) = h;
  if (a.lo) {
    float hf[8], r[8];
    unpack8(h, hf);
#pragma unroll
    for (int i = 0; i < 8; ++i) r[i] = f[i] - hf[i];
    *reinterpret_cast<uint4*>(q + a.lo) = pack8(r);
  }
}

// ------------------------------------------------------------------------------------------------
// Programmatic dependent launch (PDL).  Every kernel calls pdl_wait() before touching memory written by the
// previous kernel in the stream and pdl_launch() as early as possible, so that the launch latency and the
// prologue of kernel k+1 overlap the execution of kernel k.  Without the launch attribute both are no-ops.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

bool pdl_enabled();            // FPNMT_OPT_NO_PDL disables the launch attribute (api.cu)
void set_pdl_enabled(bool on);   // process-wide; Engine::init sets it from fpnmt_config.kernel_opts

template <typename... KArgs, typename... Args>
inline cudaError_t launch_k_pdl(bool pdl, void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream,
                                Args... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = pdl ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}
template <typename... KArgs, typename... Args>
inline cudaError_t launch_k(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream,
                            Args... args) {
  return launch_k_pdl(pdl_enabled(), kernel, grid, block, smem, stream, args...);
}

// ------------------------------------------------------------------------------------------------
// warp helpers
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ bool elect_one() {
  uint32_t pred = 0;
  asm volatile(
      "{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}\n"
      : "=r"(pred));
  return pred != 0;
}

// ------------------------------------------------------------------------------------------------
// mbarrier
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "WAIT_%=:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra DONE_%=;\n\t"
      "bra WAIT_%=;\n\t"
      "DONE_%=:\n\t}\n" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// ------------------------------------------------------------------------------------------------
// TMA (cp.async.bulk.tensor), tile mode, completion on an mbarrier
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(m) : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* smem, const CUtensorMap* m, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
          smem_u32(smem)),
      "l"(m), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_load_4d(void* smem, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2,
                                            int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], "
      "[%2];" ::"r"(smem_u32(smem)),
      "l"(m), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}

// ------------------------------------------------------------------------------------------------
// tcgen05 / TMEM
// ------------------------------------------------------------------------------------------------
template <int COLS>
__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "n"(COLS)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
template <int COLS>
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(COLS) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// D[tmem] (+)= A[smem desc] * B[smem desc], bf16 inputs, fp32 accumulate, issued by ONE thread.
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}\n" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Predicated forms for a CONVERGENT issuing warp: all 32 lanes execute the surrounding (uniform) control flow and only the
// lane with `pred != 0` issues.  Inside an `if (lane == 0)` region ptxas has to move every non-provably-uniform operand
// (e.g. the TMEM address read from shared memory) into a uniform register with an ELECT / R2UR.BROADCAST retry loop in
// front of EVERY tcgen05.mma (9 extra instructions and ~50 cycles per MMA on the single issuing thread).
__device__ __forceinline__ void umma_bf16_pred(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate,
                                               uint32_t pred) {
  asm volatile(
      "{\n\t.reg .pred p, q;\n\tsetp.ne.b32 p, %4, 0;\n\tsetp.ne.b32 q, %5, 0;\n\t"
      "@q tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}\n" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate), "r"(pred)
      : "memory");
}
__device__ __forceinline__ void umma_commit_pred(uint64_t* bar, uint32_t pred) {
  asm volatile(
      "{\n\t.reg .pred q;\n\tsetp.ne.b32 q, %1, 0;\n\t"
      "@q tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n\t}\n" ::"r"(smem_u32(bar)), "r"(pred)
      : "memory");
}
__device__ __forceinline__ void tma_load_2d_pred(void* smem, const CUtensorMap* m, uint64_t* bar, int c0, int c1, uint32_t pred) {
  asm volatile(
      "{\n\t.reg .pred q;\n\tsetp.ne.b32 q, %5, 0;\n\t"
      "@q cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];\n\t}\n" ::"r"(
          smem_u32(smem)),
      "l"(m), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(pred)
      : "memory");
}
__device__ __forceinline__ void tma_load_4d_pred(void* smem, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2, int c3,
                                                 uint32_t pred) {
  asm volatile(
      "{\n\t.reg .pred q;\n\tsetp.ne.b32 q, %7, 0;\n\t"
      "@q cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];\n\t}\n" ::"r"(
          smem_u32(smem)),
      "l"(m), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(pred)
      : "memory");
}
__device__ __forceinline__ void mbar_expect_tx_pred(uint64_t* bar, uint32_t bytes, uint32_t pred) {
  asm volatile(
      "{\n\t.reg .pred q;\n\tsetp.ne.b32 q, %2, 0;\n\t"
      "@q mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n\t}\n" ::"r"(smem_u32(bar)), "r"(bytes), "r"(pred)
      : "memory");
}
// Arrive on an mbarrier when all previously issued tcgen05.mma of this thread have completed.
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}
// 32 lanes x 32 consecutive fp32 columns: thread i of the warp receives lane (base_lane + i).
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t* r) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// Shared-memory matrix descriptor for a K-major bf16 tile whose rows are 128 bytes (64 elements)
// laid out by TMA with CU_TENSOR_MAP_SWIZZLE_128B: 8-row groups are 1024 B apart (SBO), LBO unused,
// descriptor version 1 (sm_100), layout type 2 = SWIZZLE_128B.  `addr` must be 1024 B aligned
// (+ k*32 B to step UMMA_K=16 elements inside the swizzle atom).
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3ffffu) >> 4);   // start address, 16 B units, bits [0,14)
  d |= (uint64_t)1 << 16;                         // leading byte offset (ignored for swizzled K-major)
  d |= (uint64_t)(1024 >> 4) << 32;               // stride byte offset = 1024 B, bits [32,46)
  d |= (uint64_t)1 << 46;                         // descriptor version (sm_100)
  d |= (uint64_t)2 << 61;                         // SWIZZLE_128B
  return d;
}
// Instruction descriptor, kind::f16: bf16 x bf16 -> fp32, both operands K-major, M x N tile.
__host__ __device__ constexpr uint32_t umma_idesc_bf16(int m, int n) {
  return (1u << 4)                      // c_format = F32
         | (1u << 7)                    // a_format = BF16
         | (1u << 10)                   // b_format = BF16
         | ((uint32_t)(n >> 3) << 17)   // n_dim
         | ((uint32_t)(m >> 4) << 24);  // m_dim
}

}  // namespace fpnmt
