// Device-side helpers shared by every kernel of libhqgraft: sm_100a PTX wrappers (mbarrier, TMA,
// tcgen05 / TMEM), vector loads, warp reductions, Philox4x32-10.
#pragma once

#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <type_traits>

namespace hq {

typedef __nv_bfloat16 bf16;
typedef __half f16;   // IEEE binary16: the element type of the HQ_PREC_F16 engine

// ------------------------------------------------------------------------------------------------
// small utilities
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

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

template <typename T> struct ActT;
template <> struct ActT<float> {
  static __device__ __forceinline__ float to_f(float v) { return v; }
  static __device__ __forceinline__ float from_f(float v) { return v; }
};
template <> struct ActT<bf16> {
  static __device__ __forceinline__ float to_f(bf16 v) { return __bfloat162float(v); }
  static __device__ __forceinline__ bf16 from_f(float v) { return __float2bfloat16_rn(v); }
};
template <> struct ActT<f16> {
  static __device__ __forceinline__ float to_f(f16 v) { return __half2float(v); }
  static __device__ __forceinline__ f16 from_f(float v) { return __float2half_rn(v); }
};

// Two fp32 values rounded to nearest-even into one 32-bit pair of a 2-byte type (low half = a), and back.
template <typename AT> __device__ __forceinline__ uint32_t pack2_rn(float a, float b);
template <> __device__ __forceinline__ uint32_t pack2_rn<bf16>(float a, float b) {
  __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&h);
}
template <> __device__ __forceinline__ uint32_t pack2_rn<f16>(float a, float b) {
  __half2 h = __floats2half2_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&h);
}
template <typename AT> __device__ __forceinline__ float2 unpack2(uint32_t u);
template <> __device__ __forceinline__ float2 unpack2<bf16>(uint32_t u) {
  return __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&u));
}
template <> __device__ __forceinline__ float2 unpack2<f16>(uint32_t u) {
  return __half22float2(*reinterpret_cast<const __half2*>(&u));
}

// 8 consecutive activations -> fp32 (16-byte load for bf16, 2x16 for fp32). p must be 16B aligned.
__device__ __forceinline__ void load8(const bf16* p, float (&o)[8]) {
  uint4 u = *reinterpret_cast<const uint4*>(p);
  const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&u);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    float2 f = __bfloat1622float2(h[i]);
    o[2 * i] = f.x;
    o[2 * i + 1] = f.y;
  }
}
__device__ __forceinline__ void load8(const f16* p, float (&o)[8]) {
  uint4 u = *reinterpret_cast<const uint4*>(p);
  const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float2 f = unpack2<f16>(w[i]);
    o[2 * i] = f.x;
    o[2 * i + 1] = f.y;
  }
}
__device__ __forceinline__ void load8(const float* p, float (&o)[8]) {
  float4 a = *reinterpret_cast<const float4*>(p);
  float4 b = *reinterpret_cast<const float4*>(p + 4);
  o[0] = a.x; o[1] = a.y; o[2] = a.z; o[3] = a.w;
  o[4] = b.x; o[5] = b.y; o[6] = b.z; o[7] = b.w;
}
// streaming variant (read once: KV cache) - bypass L1 allocation
__device__ __forceinline__ void load8_stream(const bf16* p, float (&o)[8]) {
  uint4 u;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
               : "=r"(u.x), "=r"(u.y), "=r"(u.z), "=r"(u.w) : "l"(p));
  const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&u);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    float2 f = __bfloat1622float2(h[i]);
    o[2 * i] = f.x;
    o[2 * i + 1] = f.y;
  }
}
__device__ __forceinline__ void load8_stream(const f16* p, float (&o)[8]) {
  uint4 u;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
               : "=r"(u.x), "=r"(u.y), "=r"(u.z), "=r"(u.w) : "l"(p));
  const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float2 f = unpack2<f16>(w[i]);
    o[2 * i] = f.x;
    o[2 * i + 1] = f.y;
  }
}
__device__ __forceinline__ void load8_stream(const float* p, float (&o)[8]) { load8(p, o); }

__device__ __forceinline__ void store8(bf16* p, const float (&v)[8]) {
  uint4 u;
  __nv_bfloat162* h = reinterpret_cast<__nv_bfloat162*>(&u);
#pragma unroll
  for (int i = 0; i < 4; ++i) h[i] = __floats2bfloat162_rn(v[2 * i], v[2 * i + 1]);
  *reinterpret_cast<uint4*>(p) = u;
}
__device__ __forceinline__ void store8(f16* p, const float (&v)[8]) {
  *reinterpret_cast<uint4*>(p) = make_uint4(pack2_rn<f16>(v[0], v[1]), pack2_rn<f16>(v[2], v[3]), pack2_rn<f16>(v[4], v[5]),
                                            pack2_rn<f16>(v[6], v[7]));
}
__device__ __forceinline__ void store8(float* p, const float (&v)[8]) {
  *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
  *reinterpret_cast<float4*>(p + 4) = make_float4(v[4], v[5], v[6], v[7]);
}

// ------------------------------------------------------------------------------------------------
// Philox4x32-10 (Salmon et al., SC'11) - counter-based RNG for the categorical draws
// ------------------------------------------------------------------------------------------------
__host__ __device__ __forceinline__ void philox4x32_10(uint32_t k0, uint32_t k1, uint32_t c0, uint32_t c1,
                                                       uint32_t c2, uint32_t c3, uint32_t (&out)[4]) {
  const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    uint64_t p0 = static_cast<uint64_t>(M0) * c0;
    uint64_t p1 = static_cast<uint64_t>(M1) * c2;
    uint32_t hi0 = static_cast<uint32_t>(p0 >> 32), lo0 = static_cast<uint32_t>(p0);
    uint32_t hi1 = static_cast<uint32_t>(p1 >> 32), lo1 = static_cast<uint32_t>(p1);
    uint32_t n0 = hi1 ^ c1 ^ k0, n1 = lo1, n2 = hi0 ^ c3 ^ k1, n3 = lo0;
    c0 = n0; c1 = n1; c2 = n2; c3 = n3;
    k0 += W0; k1 += W1;
  }
  out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

// uniform in (0, 1): 23 random bits, centred ((n + 0.5) * 2^-23 is exact in fp32) so 0 and 1 never occur
__host__ __device__ __forceinline__ float u01_from_bits(uint32_t x) {
  return (static_cast<float>(x >> 9) + 0.5f) * (1.0f / 8388608.0f);
}

// Instruction descriptor for kind::f16 with bf16 A/B (both K-major), fp32 accumulate, M x N tile.
// Field layout as in cute/arch/mma_sm100_desc.hpp (InstrDescriptor).
__host__ __device__ constexpr uint32_t umma_idesc_bf16(int M, int N) {
  return (1u << 4)                               // c_format = F32
         | (1u << 7)                             // a_format = BF16
         | (1u << 10)                            // b_format = BF16
         | (static_cast<uint32_t>(N >> 3) << 17) // n_dim
         | (static_cast<uint32_t>(M >> 4) << 24);// m_dim
}
// The same with IEEE fp16 A/B: a_format = b_format = F16 (0) under kind::f16.
__host__ __device__ constexpr uint32_t umma_idesc_f16(int M, int N) {
  return (1u << 4)                               // c_format = F32
         | (static_cast<uint32_t>(N >> 3) << 17) // n_dim
         | (static_cast<uint32_t>(M >> 4) << 24);// m_dim
}
// The descriptor for operands of the 2-byte type AT (bf16 | f16)
template <typename AT>
__host__ __device__ constexpr uint32_t umma_idesc(int M, int N) {
  static_assert(std::is_same<AT, bf16>::value || std::is_same<AT, f16>::value, "kind::f16 takes bf16 or fp16 operands");
  return std::is_same<AT, bf16>::value ? umma_idesc_bf16(M, N) : umma_idesc_f16(M, N);
}
// Instruction descriptor for kind::tf32: a_format = b_format = TF32 (2), both K-major, fp32 accumulate.  The operands are
// fp32 in memory; the tensor core reads the sign, exponent and top 10 mantissa bits.
__host__ __device__ constexpr uint32_t umma_idesc_tf32(int M, int N) {
  return (1u << 4)                               // c_format = F32
         | (2u << 7)                             // a_format = TF32
         | (2u << 10)                            // b_format = TF32
         | (static_cast<uint32_t>(N >> 3) << 17) // n_dim
         | (static_cast<uint32_t>(M >> 4) << 24);// m_dim
}

// ------------------------------------------------------------------------------------------------
// Kernel timeline tracing (hq_trace_run): every loop kernel takes a launch id as its first parameter; when it is
// >= 0, thread 0 of every CTA folds %globaltimer into [min start, max end] of that launch.  id < 0: no cost.
// ------------------------------------------------------------------------------------------------
__device__ unsigned long long* g_hq_trace = nullptr;

struct TraceScope {
  int id;
  __device__ __forceinline__ explicit TraceScope(int i) : id(i) {
#if defined(__CUDA_ARCH__)
    if (id >= 0 && threadIdx.x == 0) {
      unsigned long long t;
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
      atomicMin(&g_hq_trace[2 * id], t);
    }
#endif
  }
  __device__ __forceinline__ ~TraceScope() {
#if defined(__CUDA_ARCH__)
    if (id >= 0 && threadIdx.x == 0) {
      unsigned long long t;
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
      atomicMax(&g_hq_trace[2 * id + 1], t);
    }
#endif
  }
};

// Phase timestamps inside a kernel (hq_debug_attention_phases): when the buffer is set, one thread per CTA stores
// %globaltimer at up to 8 named points of the CTA's life; the host reduces them to min / mean / max per phase.
__device__ unsigned long long* g_hq_phase = nullptr;
__device__ __forceinline__ void phase_mark(int p) {
#if defined(__CUDA_ARCH__)
  if (g_hq_phase != nullptr) {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    g_hq_phase[blockIdx.x * 8 + p] = t;
  }
#endif
}

// The same stamps for ONE launch of a traced run (hq_debug_gemm_phases): the launch whose trace id is g_hq_phase_id.
// Compiled in only with -DHQ_PHASE_STAMPS (python hqtransformer_b200/build.py --phase-stamps): a lane-dependent branch
// inside the warp-uniform producer / MMA loops costs 6 % of the whole sampling step even when it is never taken (ptxas
// falls back to the ELECT / R2UR waterfall around every UTCHMMA; 3 277 vs 3 065 images/s, profiles/r2_epilogue_ab.txt).
// (its own buffer: other kernels stamp g_hq_phase unconditionally while it is set)
__device__ int g_hq_phase_id = -1;
__device__ unsigned long long* g_hq_gemm_phase = nullptr;
__device__ __forceinline__ void phase_mark_if(bool on, int p) {
#if defined(__CUDA_ARCH__) && defined(HQ_PHASE_STAMPS)
  if (on && g_hq_gemm_phase != nullptr) {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    g_hq_gemm_phase[blockIdx.x * 16 + p] = t;
  }
#endif
}

// Programmatic dependent launch: wait for the producer grid's memory / let the dependent grid start its prologue
__device__ __forceinline__ void pdl_wait() {
#if defined(__CUDA_ARCH__)
  asm volatile("griddepcontrol.wait;" ::: "memory");
#endif
}
__device__ __forceinline__ void pdl_launch_dependents() {
#if defined(__CUDA_ARCH__)
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
#endif
}

#if defined(__CUDA_ARCH__)
// One lane of a CONVERGED warp (the same lane every time for the same mask).  The single-thread roles (TMA producer,
// tcgen05.mma issuer) run as warp-uniform code and issue under this predicate: inside `if (lane == 0)` ptxas must
// assume divergence and wraps every UTMALDG / UTCHMMA in an ELECT + R2UR.BROADCAST "waterfall" loop - measured ~77 clk
// per MMA and ~130 clk per TMA issue (profiles/r2_gemm_loop_prof.txt) - whereas operands computed in uniform control
// flow stay in uniform registers.
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n"
      ".reg .pred P;\n"
      "elect.sync _|P, 0xffffffff;\n"
      "selp.u32 %0, 1, 0, P;\n"
      "}\n"
      : "=r"(pred));
  return pred != 0;
}

// ------------------------------------------------------------------------------------------------
// mbarrier
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
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
  uint32_t done;
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
      "selp.u32 %0, 1, 0, p;\n"
      "}\n"
      : "=r"(done)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return done != 0;
}
// Waits for the phase with the given parity to complete (plain try_wait: the hardware parks the thread for a short,
// implementation-defined time per attempt and wakes it promptly on completion; an explicit suspend-time hint was
// measured to ADD ~5 us to a 13 us kernel).  A wait that needs more than ~16M attempts can only be a protocol bug:
// trap instead of hanging the GPU.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t polls = 0;
  while (!mbar_try_wait(bar, parity)) {
    if (++polls > (1u << 24)) __trap();
  }
}
// Waits for two barriers at once: both try_wait requests are in flight together, so a thread that needs two operands
// (the A and the W ring of the pair GEMM) pays one ~200-clk barrier round trip per stage, not two.
__device__ __forceinline__ void mbar_wait2(uint64_t* bar1, uint32_t parity1, uint64_t* bar2, uint32_t parity2) {
  uint32_t polls = 0;
  bool d1 = false, d2 = false;
  while (true) {
    const bool t1 = d1 || mbar_try_wait(bar1, parity1);
    const bool t2 = d2 || mbar_try_wait(bar2, parity2);
    d1 = t1;
    d2 = t2;
    if (d1 && d2) break;
    if (++polls > (1u << 24)) __trap();
  }
}
// Polling with back-off for waits whose wake-up latency is not critical (consumers of a deep ring that many warps
// of many resident CTAs poll at once): the sleeping warp frees issue slots for the warps that have data.
__device__ __forceinline__ void mbar_wait_sleep(uint64_t* bar, uint32_t parity, unsigned ns) {
  uint32_t polls = 0;
  while (!mbar_try_wait(bar, parity)) {
    __nanosleep(ns);
    if (++polls > (1u << 24)) __trap();
  }
}

// ------------------------------------------------------------------------------------------------
// TMA (cp.async.bulk.tensor) - 2D tile load global -> shared, completion on an mbarrier
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d(void* smem_dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
// 1D bulk copy global -> shared (contiguous bytes; multiple of 16, 16B-aligned both sides)
__device__ __forceinline__ void bulk_load_1d(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
      ::"r"(smem_u32(smem_dst)), "l"(gsrc), "r"(bytes), "r"(smem_u32(bar))
      : "memory");
}

// ------------------------------------------------------------------------------------------------
// tcgen05 / TMEM
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_result, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_result)),
               "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// D[tmem] (+)= A[smem] * B[smem]^T, bf16 x bf16 (or fp16 x fp16, as the descriptor says) -> fp32; issued by ONE thread
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrive on an mbarrier once every tcgen05.mma issued so far by this thread has completed
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}
// 32 lanes x 32 consecutive fp32 columns: thread i of the warp receives row (lane base + i)
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,"
      "%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// Shared-memory matrix descriptor for a K-major bf16 tile whose rows are 128 bytes (64 elements),
// written by TMA with CU_TENSOR_MAP_SWIZZLE_128B: 8-row groups are 1024 B apart (SBO), LBO unused,
// descriptor version 1 (sm_100), layout type 2 (SWIZZLE_128B).  Field layout as in
// cute/arch/mma_sm100_desc.hpp (SmemDescriptor).
__device__ __forceinline__ uint64_t umma_smem_desc_sw128(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr & 0x3FFFFu) >> 4);  // start address, bits [0,14)
  d |= static_cast<uint64_t>(0) << 16;                       // leading byte offset (ignored for swizzled K-major)
  d |= static_cast<uint64_t>(1024 >> 4) << 32;               // stride byte offset, bits [32,46)
  d |= static_cast<uint64_t>(1) << 46;                       // version = 1
  d |= static_cast<uint64_t>(2) << 61;                       // SWIZZLE_128B
  return d;
}


// ------------------------------------------------------------------------------------------------
// CTA pairs (cta_group::2): both CTAs of a 2-CTA cluster feed one tcgen05.mma of M = 256.
// PTX forms as in cute/arch/copy_sm100_tma.hpp (SM100_TMA_2SM_LOAD_2D), cute/arch/tmem_allocator_sm100.hpp
// (Allocator2Sm) and cutlass/arch/barrier.h (umma_arrive_multicast_2x1SM).
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// Execution barrier only (no memory ordering): for a tear-down in which nothing written by this thread is read by the peer
// afterwards.  The release form makes every thread wait for its global stores to drain before it may arrive.
__device__ __forceinline__ void cluster_sync_relaxed() {
  asm volatile("barrier.cluster.arrive.relaxed.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.aligned;" ::: "memory");
}
// TMA tile load into THIS CTA's shared memory whose transaction bytes are credited to the mbarrier at the same
// offset in the pair's leader CTA (peer bit of the shared::cluster address cleared).
__device__ __forceinline__ void tma_load_2d_2sm(void* smem_dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar) & 0xFEFFFFFFu), "r"(c0), "r"(c1)
      : "memory");
}
// 3-D form: the GEMM operands viewed as [K / 64][rows][64] so that ONE instruction stages several 64-wide k-blocks
__device__ __forceinline__ void tma_load_3d_2sm(void* smem_dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar) & 0xFEFFFFFFu), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
__device__ __forceinline__ void tmem_alloc_2sm(uint32_t* smem_result, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_result)),
               "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish_2sm() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_2sm(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// D[tmem of both CTAs] (+)= A (128 rows from each CTA) * B^T (N/2 rows from each CTA); issued by ONE thread of the leader
__device__ __forceinline__ void umma_bf16_2sm(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                              uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// The same with tf32 x tf32 -> fp32 (kind::tf32, K = 8 per instruction: 32 bytes of a K-major row, as K = 16 of bf16)
__device__ __forceinline__ void umma_tf32_2sm(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                              uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::2.kind::tf32 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrive on the mbarrier at this offset in every CTA of `cta_mask` once all prior tcgen05.mma of this thread completed
__device__ __forceinline__ void umma_commit_2sm(uint64_t* bar, uint16_t cta_mask) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
               ::"r"(smem_u32(bar)), "h"(cta_mask)
               : "memory");
}
#endif  // __CUDA_ARCH__

}  // namespace hq
