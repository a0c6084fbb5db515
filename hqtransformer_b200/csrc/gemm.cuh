// GEMM family of libhqgraft: C[M,N] = A[M,K] * W[N,K]^T with fused epilogues.
//
//   gemm_tc_kernel    bf16 x bf16 (or fp16 x fp16: AT) -> fp32 on the 5th-gen tensor cores: TMA (SWIZZLE_128B) stages A and W
//                     tiles into a ring of shared-memory slots, one thread issues tcgen05.mma with the
//                     accumulator in TMEM, four warps drain TMEM with tcgen05.ld and apply the epilogue.
//   gemm_simt_kernel  fp32 on CUDA cores, for HQ_PREC_FP32 (the reference's use_fp16=False path).
//
// Epilogues replace the separate ATen ops of the reference (SURVEY.md 2b K3/K4/K7/K8/K9):
//   EPI_QKV    + bias; q -> [M, D] activation buffer, k / v -> straight into their KV-cache slot
//              (layers.py:73, 84-96: three addmm + stack + cat)
//   EPI_RESID  x += acc + bias                (layers.py:190 + :326/:327 residual adds)
//   EPI_GELU   out = gelu_erf(acc + bias)     (layers.py:312-314)
//   EPI_F32    out = acc                      (head_top / head_bot, hierarchical_ar.py:695, 715)
//   EPI_SAMPLE head + Sample(z; T, None, None) (hierarchical_ar.py:695 / 715 + 762-785 with no top-k / top-p cut): the
//              [rows, V] logits never leave the SM - see epilogue_sample_tile
#pragma once

#include "common.cuh"
#include "../../include/hqgraft.h"

namespace hq {

enum { EPI_QKV = 0, EPI_RESID = 1, EPI_GELU = 2, EPI_F32 = 3, EPI_SAMPLE = 4 };

template <typename AT>
struct EpiParams {
  const float* bias;  // [N] fp32 or nullptr
  // EPI_QKV: column n belongs to section sec0 + n / D (0 = q, 1 = k, 2 = v)
  AT* q;              // [M, D]
  AT* kdst;           // rows of D; row index = (m / rpb) * t_stride + t0 + (m % rpb)
  AT* vdst;
  AT* vdup;           // optional second copy of the v rows as [M, D] (depth pass 0: attention output == v)
  int D, sec0, rpb, t_stride, t0;
  // EPI_RESID
  float* x;           // [M, N] fp32, read-modify-write
  // EPI_GELU
  AT* out;            // [M, N]
  // EPI_F32
  float* outf;        // [M, ldo]; split-K: slice blockIdx.z of the K range writes outf + blockIdx.z * split_stride
  int ldo;
  size_t split_stride;
  // EPI_SAMPLE
  const hq_sampling_params* sp;   // device copy (temperature, seed, row offset)
  float2* samp_part;              // [M, N / 32]: per 32-column chunk (log-sum-exp, index drawn inside the chunk as int bits)
  int temp_sel, rows_per_b, slot0, pos;
  // debug (hq_bench_gemm_shape with HQ_GEMM_PROF): clock64 sums of the producer / MMA-issuer loops of pair 0's leader
  long long* prof;
  long long prof_pad;   // keeps sizeof(EpiParams) (and the chain kernel's ChainOp) a multiple of 16
};


__device__ __forceinline__ float gelu_erf(float v) { return 0.5f * v * (1.0f + erff(v * 0.70710678118654752440f)); }

// The same function for outputs that are rounded to a 2-byte type (the tcgen05 engines, bf16 and fp16): x * Phi(x) with
// Phi(x) = 1 - erfc(|x| / sqrt 2) / 2 (x >= 0), erfc(|x| / sqrt 2) / 2 (x < 0) and erfc by Abramowitz & Stegun 7.1.26
// (|error| <= 1.5e-7 on erfc): one rcp, one ex2 and a degree-5 Horner form, ~15 instructions against ~35 for erff.  The
// bound is absolute: |gelu_bf16out(x) - gelu(x)| <= ~4.3e-7 over [-12, 12] (fp32 restatement), below half a bf16 ulp of
// the result wherever |gelu(x)| >~ 1e-4; for x < -6, where |gelu(x)| < 1e-8, the RELATIVE error reaches a few percent
// (several bf16 ulps of a value that is ~0 next to the rest of the row).  tests/test_gpu_epilogues.py holds the kernel
// to |got - gelu| <= half a bf16 ulp of gelu + 5e-7.  The same absolute bound is far below half an fp16 ulp wherever
// |gelu(x)| >~ 1e-3 (fp16 keeps 11 significant bits); tests/test_gpu_fp16.py holds the fp16 epilogue to half an fp16
// ulp + 5e-7.  The exact-erf epilogue of fc1 was issue-bound on erff: 1.1 of the
// 1.65 us per 32-column chunk, on the critical path of every fc1 launch (profiles/r2_gemm_phases.txt).  The fp32 engine
// (bit-exact parity with the reference) keeps gelu_erf.
__device__ __forceinline__ float gelu_bf16out(float v) {
  const float z = fabsf(v) * 0.70710678118654752440f;
  const float t = __fdividef(1.0f, fmaf(0.3275911f, z, 1.0f));
  float p = fmaf(1.061405429f, t, -1.453152027f);
  p = fmaf(p, t, 1.421413741f);
  p = fmaf(p, t, -0.284496736f);
  p = fmaf(p, t, 0.254829592f);
  float e;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(-1.4426950408889634f * z * z));
  const float h = 0.5f * p * t * e;                                       // erfc(z) / 2
  return v * (v >= 0.f ? 1.0f - h : h);
}
template <typename AT>
__device__ __forceinline__ float gelu_for(float v) { return sizeof(AT) == 2 ? gelu_bf16out(v) : gelu_erf(v); }

// 8 consecutive columns n0..n0+7 of row m (n0 % 8 == 0, all < N)
template <int EPI, typename AT>
__device__ __forceinline__ void epi_store8(const EpiParams<AT>& ep, int m, int n0, int N, float (&v)[8]) {
  if (EPI != EPI_F32 && ep.bias != nullptr) {
    const float4 b0 = *reinterpret_cast<const float4*>(ep.bias + n0);
    const float4 b1 = *reinterpret_cast<const float4*>(ep.bias + n0 + 4);
    v[0] += b0.x; v[1] += b0.y; v[2] += b0.z; v[3] += b0.w;
    v[4] += b1.x; v[5] += b1.y; v[6] += b1.z; v[7] += b1.w;
  }
  if (EPI == EPI_QKV) {
    const int sec = ep.sec0 + n0 / ep.D;
    const int c = n0 % ep.D;
    if (sec == 0) {
      store8(ep.q + static_cast<size_t>(m) * ep.D + c, v);
    } else {
      const size_t row = static_cast<size_t>(m / ep.rpb) * ep.t_stride + ep.t0 + (m % ep.rpb);
      AT* dst = (sec == 1 ? ep.kdst : ep.vdst) + row * ep.D + c;
      store8(dst, v);
      if (sec == 2 && ep.vdup != nullptr) store8(ep.vdup + static_cast<size_t>(m) * ep.D + c, v);
    }
  } else if (EPI == EPI_RESID) {
    float* p = ep.x + static_cast<size_t>(m) * N + n0;
    float4 a = *reinterpret_cast<float4*>(p);
    float4 b = *reinterpret_cast<float4*>(p + 4);
    a.x += v[0]; a.y += v[1]; a.z += v[2]; a.w += v[3];
    b.x += v[4]; b.y += v[5]; b.z += v[6]; b.w += v[7];
    *reinterpret_cast<float4*>(p) = a;
    *reinterpret_cast<float4*>(p + 4) = b;
  } else if (EPI == EPI_GELU) {
#pragma unroll
    for (int i = 0; i < 8; ++i) v[i] = gelu_erf(v[i]);
    store8(ep.out + static_cast<size_t>(m) * N + n0, v);
  } else {
    store8(ep.outf + static_cast<size_t>(m) * ep.ldo + n0, v);
  }
}


// ------------------------------------------------------------------------------------------------
// Epilogue of the tcgen05 kernels.  tcgen05.ld hands every thread one ROW of the accumulator, which would make each
// global store touch 32 different lines (half-written sectors: measured 1.6 us for a 128 x 64 tile and 6.7 us for
// 128 x 256, profiles/r1_gemm_trace.txt).  Instead each warp parks its 32 x 32 fp32 chunk in a private 4 KB slab of
// shared memory (the finished pipeline's stage-0 buffer; 16-byte pieces XOR-swizzled by row so both phases are
// bank-conflict free) and writes it out with 8 lanes per row: every store instruction covers 4 complete 128-byte row
// pieces (64-byte pieces for bf16 outputs).  Bias / GELU / residual are applied at write-out.
// ------------------------------------------------------------------------------------------------
#if defined(__CUDA_ARCH__)
// `sbias` points at BN floats of shared memory outside the pipeline stages (filled here, before the accumulator is
// complete, so the cold bias loads overlap the main loop).  The chunk loop is NOT unrolled and all index arithmetic
// (section of the fused q/k/v columns, KV-cache row of each output row) is hoisted: the epilogue is straight-line code
// that every warp fetches once per launch, and a decode step launches ~80 GEMMs with a cold instruction cache.
// NW = 4: one warp per TMEM lane quarter (warp % 4).  NW = 8 (pair kernel): two warps per quarter, `half` = 0 / 1 taking
// the even / odd 32-column chunks - the epilogue (tcgen05.ld, smem transpose, bias / GELU, stores) is pure per-element
// work on the critical path of every launch, so twice the warps halve it.  `ew` = 0..NW-1 indexes the warp's slab.
template <int BN, int EPI, typename AT, int NW = 4>
__device__ __forceinline__ void epilogue_tile(uint32_t tmem_base, uint8_t* slab_base, float* sbias, int warp, int lane,
                                              int m0, int n0, int M, int N, const EpiParams<AT>& ep,
                                              uint64_t* tmem_full_bar, uint32_t full_parity = 0, int ew = -1, bool pm = false) {
  const int quarter = warp & 3;
  if (ew < 0) ew = quarter;
  const int half = ew >> 2;
  const int etid = ew * 32 + lane;                             // 0..NW*32-1 over the epilogue warps
  const bool has_bias = (EPI != EPI_F32) && ep.bias != nullptr;
  if (has_bias) {
    // persistent kernel: previous tile's bias fully consumed
    if (NW == 8) asm volatile("bar.sync 1, 256;" ::: "memory"); else asm volatile("bar.sync 1, 128;" ::: "memory");
    for (int i = etid; i < BN; i += NW * 32) sbias[i] = (n0 + i < N) ? ep.bias[n0 + i] : 0.f;
  }
  // rows this lane writes: it*4 + (lane >> 3) of the warp's 32; destination row offsets (elements) per row.
  // Computed ONCE per tile, here, while the main loop still runs, and then made opaque to the compiler: left alone,
  // nvcc re-materialised the divisions of the KV-cache row (m / rpb, m % rpb) and of the q/k/v section inside every one
  // of the 8 write-out iterations, each behind its own branch - ~180 dependent clocks per iteration, 0.7-1.7 us per
  // 32-column chunk on the critical path of EVERY GEMM launch (profiles/r2_gemm_phases.txt: parked -> stored).
  const int piece = lane & 7;
  size_t row_a[8], row_b[8];
  bool row_ok[8];
  {
    const int mbase = m0 + quarter * 32 + (lane >> 3);
    int kb = 0, kr = 0;                                          // image / row within the image of row m (EPI_QKV)
    if (EPI == EPI_QKV) {
      kb = mbase / ep.rpb;
      kr = mbase - kb * ep.rpb;
    }
#pragma unroll
    for (int it = 0; it < 8; ++it) {
      const int m = mbase + it * 4;
      row_ok[it] = m < M;
      if (EPI == EPI_QKV) {
        row_a[it] = static_cast<size_t>(m) * ep.D;                                                    // q / vdup row
        row_b[it] = (static_cast<size_t>(kb) * ep.t_stride + ep.t0 + kr) * ep.D;                      // k / v row
        kr += 4;                                                                                       // next row: m + 4
        while (kr >= ep.rpb) {
          kr -= ep.rpb;
          ++kb;
        }
      } else if (EPI == EPI_F32) {
        row_a[it] = static_cast<size_t>(m) * ep.ldo;
        row_b[it] = 0;
      } else {
        row_a[it] = static_cast<size_t>(m) * N;
        row_b[it] = 0;
      }
      asm volatile("" : "+l"(row_a[it]), "+l"(row_b[it]));
    }
  }
  // sbias visible to all epilogue warps
  if (NW == 8) asm volatile("bar.sync 1, 256;" ::: "memory"); else asm volatile("bar.sync 1, 128;" ::: "memory");
  mbar_wait(tmem_full_bar, full_parity);
  if (warp == 2 && lane == 0) phase_mark_if(pm, 5);
  tc_fence_after();

  uint8_t* slab = slab_base + ew * 4096;                       // this warp's 32 rows x 128 B
  const uint32_t slab_u32 = smem_u32(slab);
  // shared-memory addresses of this lane's 8 pieces (row it*4 + (lane >> 3), 16-byte piece XOR-swizzled by row)
  uint32_t rd_addr[8];
#pragma unroll
  for (int it = 0; it < 8; ++it) {
    const int row = it * 4 + (lane >> 3);
    rd_addr[it] = slab_u32 + row * 128 + ((piece ^ (row & 7)) << 4);
  }
#pragma unroll 1
  for (int c = (NW == 8 ? half : 0); c < BN / 32; c += (NW == 8 ? 2 : 1)) {
    uint32_t r[32];
    tmem_ld_32x32(tmem_base + (static_cast<uint32_t>(quarter * 32) << 16) + static_cast<uint32_t>(c * 32), r);
    tmem_ld_wait();
    if (warp == 2 && lane == 0 && c == 0) phase_mark_if(pm, 8);
#pragma unroll
    for (int j = 0; j < 8; ++j) {                              // row = lane; piece j -> slot j ^ (lane & 7)
      const uint32_t addr = slab_u32 + lane * 128 + ((j ^ (lane & 7)) << 4);
      asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(r[4 * j]), "r"(r[4 * j + 1]),
                   "r"(r[4 * j + 2]), "r"(r[4 * j + 3])
                   : "memory");
    }
    __syncwarp();
    if (warp == 2 && lane == 0 && c == 0) phase_mark_if(pm, 9);
    const int nb = n0 + c * 32;                                // chunk base column (a chunk never straddles q/k/v)
    const int n = nb + piece * 4;
    float4 b4 = make_float4(0.f, 0.f, 0.f, 0.f);
    if (has_bias) b4 = *reinterpret_cast<const float4*>(sbias + c * 32 + piece * 4);
    // chunk-uniform destination: base pointer of column `col`, which of the two row-offset sets, optional second copy
    AT* dst = nullptr;
    AT* dup = nullptr;
    float* dstf = nullptr;
    bool use_b = false;
    if (EPI == EPI_QKV) {
      const int s1 = nb >= ep.D ? 1 : 0, s2 = nb >= 2 * ep.D ? 1 : 0;   // section within the fused columns, no division
      const int sec = ep.sec0 + s1 + s2;
      const int col = nb - (s1 + s2) * ep.D + piece * 4;
      use_b = sec != 0;
      dst = (sec == 0 ? ep.q : (sec == 1 ? ep.kdst : ep.vdst)) + col;
      if (sec == 2 && ep.vdup != nullptr) dup = ep.vdup + col;
    } else if (EPI == EPI_GELU) {
      dst = ep.out + n;
    } else if (EPI == EPI_RESID) {
      dstf = ep.x + n;
    } else {
      dstf = ep.outf + n;
    }
    if (n < N) {
      float4 v[8];
#pragma unroll
      for (int it = 0; it < 8; ++it)
        asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v[it].x), "=f"(v[it].y), "=f"(v[it].z), "=f"(v[it].w) : "r"(rd_addr[it]));
      if (EPI == EPI_RESID) {
        float4 x4[8];
#pragma unroll
        for (int it = 0; it < 8; ++it)
          if (row_ok[it]) x4[it] = *reinterpret_cast<const float4*>(dstf + row_a[it]);
#pragma unroll
        for (int it = 0; it < 8; ++it) {
          if (row_ok[it]) {
            float4 a = x4[it];
            a.x += v[it].x + b4.x; a.y += v[it].y + b4.y; a.z += v[it].z + b4.z; a.w += v[it].w + b4.w;
            *reinterpret_cast<float4*>(dstf + row_a[it]) = a;
          }
        }
      } else {
#pragma unroll
        for (int it = 0; it < 8; ++it) {
          float4 w = v[it];
          w.x += b4.x; w.y += b4.y; w.z += b4.z; w.w += b4.w;
          if (EPI == EPI_GELU) {
            w.x = gelu_for<AT>(w.x); w.y = gelu_for<AT>(w.y); w.z = gelu_for<AT>(w.z); w.w = gelu_for<AT>(w.w);
          }
          if (EPI == EPI_F32) {
            if (row_ok[it]) *reinterpret_cast<float4*>(dstf + row_a[it]) = w;
          } else {
            const size_t ro = use_b ? row_b[it] : row_a[it];
            if constexpr (sizeof(AT) == 4) {
              if (row_ok[it]) *reinterpret_cast<float4*>(dst + ro) = w;
              if (row_ok[it] && dup != nullptr) *reinterpret_cast<float4*>(dup + row_a[it]) = w;
            } else {
              uint2 u;
              u.x = pack2_rn<AT>(w.x, w.y);
              u.y = pack2_rn<AT>(w.z, w.w);
              if (row_ok[it]) *reinterpret_cast<uint2*>(dst + ro) = u;
              if (row_ok[it] && dup != nullptr) *reinterpret_cast<uint2*>(dup + row_a[it]) = u;
            }
          }
        }
      }
    }
    __syncwarp();
    if (warp == 2 && lane == 0 && c == 0) phase_mark_if(pm, 10);
  }
}
#endif

// ------------------------------------------------------------------------------------------------
// EPI_SAMPLE: the categorical draw of Sample(z; T, None, None) without materialising the logits.  Exact two-stage sampling
// over 32-column chunks (one tcgen05.ld: thread = row, 32 consecutive logits in registers):
//   stage 1 (here): chunk c of row m -> L_c = log sum_j exp(z_j / T) and ONE index drawn inside the chunk from
//                   softmax(z_chunk / T) by inverse CDF with its own Philox uniform;
//   stage 2 (sample_finalize_kernel): chunk drawn from softmax(L) with one more uniform; the code is that chunk's index.
// P(i) = P(chunk) P(i | chunk) = exp(z_i / T) / sum exp(z / T).  Every (row, chunk) result depends only on that chunk's 32
// accumulators and on a Philox counter made of (global row, position, slot, chunk): independent of the tile shape, of the
// kernel (pair / single-CTA) and of how the batch is sharded over GPUs.
// Philox counters: (row, row >> 32, pos | (chunk / 4 + 1) << 16, slot | 0x200) -> uniform [chunk % 4] for stage 1,
//                  (row, row >> 32, pos, slot | 0x100) -> [0] for stage 2; the unfused sampler uses (row, ., pos, slot).
// ------------------------------------------------------------------------------------------------
#if defined(__CUDA_ARCH__)
template <int BN, typename AT, int NW>
__device__ __forceinline__ void epilogue_sample_tile(uint32_t tmem_base, int warp, int lane, int m0, int n0, int M, int N,
                                                     const EpiParams<AT>& ep, uint64_t* tmem_full_bar, uint32_t full_parity,
                                                     int ew) {
  const int quarter = warp & 3;
  if (ew < 0) ew = quarter;
  const int half = ew >> 2;
  const int m = m0 + quarter * 32 + lane;
  const hq_sampling_params* sp = ep.sp;
  const float temperature = ep.temp_sel == 0 ? sp->temperature_top : (ep.temp_sel == 1 ? sp->temperature_bot : sp->temperature_mid);
  const float inv_t = 1.0f / temperature;
  const uint64_t seed = sp->seed;
  const int b = m / ep.rows_per_b;
  const uint32_t slot = static_cast<uint32_t>(ep.slot0 + (m - b * ep.rows_per_b)) | 0x200u;
  const uint64_t grow = sp->row_offset + static_cast<uint64_t>(b);
  const int n_chunks = N >> 5;
  mbar_wait(tmem_full_bar, full_parity);
  tc_fence_after();
  uint32_t rnd[4] = {0u, 0u, 0u, 0u};
  int rnd_grp = -1;
#pragma unroll 1
  for (int c = (NW == 8 ? half : 0); c < BN / 32; c += (NW == 8 ? 2 : 1)) {
    uint32_t r[32];
    tmem_ld_32x32(tmem_base + (static_cast<uint32_t>(quarter * 32) << 16) + static_cast<uint32_t>(c * 32), r);
    const int gc = (n0 >> 5) + c;                               // chunk index within the row
    if ((gc >> 2) != rnd_grp) {
      rnd_grp = gc >> 2;
      philox4x32_10(static_cast<uint32_t>(seed), static_cast<uint32_t>(seed >> 32), static_cast<uint32_t>(grow),
                    static_cast<uint32_t>(grow >> 32), static_cast<uint32_t>(ep.pos) | (static_cast<uint32_t>(rnd_grp + 1) << 16),
                    slot, rnd);
    }
    const int sel = gc & 3;
    const float u = u01_from_bits(sel == 0 ? rnd[0] : (sel == 1 ? rnd[1] : (sel == 2 ? rnd[2] : rnd[3])));
    tmem_ld_wait();
    float cm = -INFINITY;
#pragma unroll
    for (int j = 0; j < 32; ++j) {
      const float z = __uint_as_float(r[j]) * inv_t;
      r[j] = __float_as_uint(z);
      cm = fmaxf(cm, z);
    }
    float run = 0.f;
#pragma unroll
    for (int j = 0; j < 32; ++j) {                              // r[j] <- inclusive prefix of exp(z - max), index order
      run += __expf(__uint_as_float(r[j]) - cm);
      r[j] = __float_as_uint(run);
    }
    const float target = u * run;
    int idx = 0;
#pragma unroll
    for (int j = 0; j < 32; ++j) idx += (__uint_as_float(r[j]) <= target) ? 1 : 0;   // first j whose prefix exceeds the target
    idx = idx > 31 ? 31 : idx;
    if (m < M)
      ep.samp_part[static_cast<size_t>(m) * n_chunks + gc] = make_float2(cm + logf(run), __int_as_float(n0 + c * 32 + idx));
  }
}
#endif

// ------------------------------------------------------------------------------------------------
// tcgen05 / TMA GEMM.  One CTA computes a 128 x BN tile; grid = (ceil(N/BN), ceil(M/128)).
//   warp 0: TMA producer (one lane)      warp 1: tcgen05.mma issuer (one lane)
//   warps 2-5: epilogue (TMEM lane quarter = warp % 4); warp 2 also owns the TMEM allocation
// tmA: A as a [rows_pad, K] bf16 tensor, box {64, 128}; tmW: W as [N_pad, K], box {64, 64}; both SWIZZLE_128B.
// ------------------------------------------------------------------------------------------------
// KS = 64-wide k-blocks per ring stage (see Tc2Cfg): KS = 2 takes 3-D boxes - tmA box {64, 128, 2}, tmW box {64, BN, 2}
// (the pair maps of width 2 * BN) - one instruction per operand and stage.
template <int BN, int KS = 1>
struct TcCfg {
  static constexpr int BM = 128, BK = 64;
  static constexpr int A_ATOM = BM * BK * 2;   // 16 KB
  static constexpr int B_ATOM = BN * BK * 2;
  static constexpr int A_BYTES = KS * A_ATOM;
  static constexpr int B_BYTES = KS * B_ATOM;
  // 144-192 KB: ONE GEMM CTA per SM (see Tc2Cfg)
  static constexpr int STAGES = KS == 1 ? ((BN == 128) ? 5 : 6) : ((BN == 128) ? 3 : 4);
  static constexpr int TMEM_COLS = BN < 32 ? 32 : BN;
  static constexpr int SMEM_BYTES = STAGES * (A_BYTES + B_BYTES) + 1024 /*align slack*/ + 256 /*barriers*/ + 1024 /*bias*/;
  static_assert(SMEM_BYTES <= 232448, "shared memory per CTA");
};

template <int BN, int EPI, typename AT, int KS = 1>
__global__ void __launch_bounds__(192, 1)
gemm_tc_kernel(int trace_id, const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmW, int M, int N, int K,
               int w_row_off, EpiParams<AT> ep) {
#if defined(__CUDA_ARCH__)
  TraceScope trace_scope(trace_id);
  using C = TcCfg<BN, KS>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~static_cast<uintptr_t>(1023));
  uint8_t* sA = smem;
  uint8_t* sB = smem + C::STAGES * C::A_BYTES;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(sB + C::STAGES * C::B_BYTES);
  uint64_t* empty_bar = full_bar + C::STAGES;
  uint64_t* tmem_full_bar = empty_bar + C::STAGES;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_full_bar + 1);
  float* sbias = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(full_bar) + 256);

  const int warp = __shfl_sync(0xffffffffu, static_cast<int>(threadIdx.x >> 5), 0);   // provably warp-uniform (role dispatch)
  const int lane = threadIdx.x & 31;
  const int m0 = blockIdx.y * C::BM;
  const int n0 = blockIdx.x * BN;
  const int num_kb = (K / C::BK) / static_cast<int>(gridDim.z);        // split-K: this CTA's share of the k-blocks
  const int num_st = (num_kb + KS - 1) / KS;                           // ring stages (the last may be short)
  const int kb0 = static_cast<int>(blockIdx.z) * num_kb;
  if (EPI == EPI_F32) ep.outf += static_cast<size_t>(blockIdx.z) * ep.split_stride;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmW);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < C::STAGES; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    mbar_init(tmem_full_bar, 1);
    fence_barrier_init();
  }
  if (warp == 2) {
    tmem_alloc(tmem_slot, C::TMEM_COLS);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  pdl_launch_dependents();
  if (warp == 0) {
    // ---- TMA producer (warp-uniform loop, one elected lane issues: see elect_one).  Weights do not depend on the
    //      previous kernel: the first ring of W tiles is requested before griddepcontrol.wait, the activation tiles
    //      after it. ----
    auto load_a = [&](int st, int slot) {
      if (KS == 1) tma_load_2d(sA + slot * C::A_BYTES, &tmA, &full_bar[slot], (kb0 + st) * C::BK, m0);
      else tma_load_3d(sA + slot * C::A_BYTES, &tmA, &full_bar[slot], 0, m0, kb0 + st * KS);
    };
    auto load_w = [&](int st, int slot) {
      if (KS == 1) {
#pragma unroll
        for (int j = 0; j < BN / 64; ++j)
          tma_load_2d(sB + slot * C::B_BYTES + j * (64 * 128), &tmW, &full_bar[slot], (kb0 + st) * C::BK, w_row_off + n0 + j * 64);
      } else {
        tma_load_3d(sB + slot * C::B_BYTES, &tmW, &full_bar[slot], 0, w_row_off + n0, kb0 + st * KS);
      }
    };
    const int pre = num_st < C::STAGES ? num_st : C::STAGES;
    if (elect_one()) {
      for (int st = 0; st < pre; ++st) {
        mbar_arrive_expect_tx(&full_bar[st], C::A_BYTES + C::B_BYTES);
        load_w(st, st);
      }
    }
    pdl_wait();
    if (elect_one()) {
      for (int st = 0; st < pre; ++st) load_a(st, st);
    }
    for (int st = pre; st < num_st; ++st) {
      const int s = st % C::STAGES;
      const uint32_t ph = (st / C::STAGES) & 1;
      mbar_wait(&empty_bar[s], ph ^ 1);
      if (elect_one()) {
        mbar_arrive_expect_tx(&full_bar[s], C::A_BYTES + C::B_BYTES);
        load_a(st, s);
        load_w(st, s);
      }
    }
  } else if (warp == 1) {
    // ---- MMA issuer (warp-uniform loop, the elected lane issues the MMAs and their commits) ----
    constexpr uint32_t idesc = umma_idesc<AT>(C::BM, BN);
    const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem_base, 0);
    for (int st = 0; st < num_st; ++st) {
      const int s = st % C::STAGES;
      const uint32_t ph = (st / C::STAGES) & 1;
      mbar_wait(&full_bar[s], ph);
      tc_fence_after();
      if (elect_one()) {
#pragma unroll
        for (int j = 0; j < KS; ++j) {
          if (KS > 1 && st * KS + j >= num_kb) break;        // short last stage
          const uint64_t da = umma_smem_desc_sw128(smem_u32(sA + s * C::A_BYTES + j * C::A_ATOM));
          const uint64_t db = umma_smem_desc_sw128(smem_u32(sB + s * C::B_BYTES + j * C::B_ATOM));
#pragma unroll
          for (int k = 0; k < C::BK / 16; ++k) {
            // advance 16 elements (32 bytes) along K inside the 128-byte swizzle atom: +2 in the >>4 address field
            umma_bf16(tmem_u, da + static_cast<uint64_t>(2 * k), db + static_cast<uint64_t>(2 * k), idesc,
                      (st > 0 || j > 0 || k > 0) ? 1u : 0u);
          }
        }
        umma_commit(&empty_bar[s]);  // frees the smem slot once these MMAs have read it
      }
    }
    if (elect_one()) umma_commit(tmem_full_bar);    // accumulator complete
  } else {
    // ---- epilogue: TMEM -> registers -> warp-private smem slab -> coalesced global ----
    pdl_wait();
    if (EPI == EPI_SAMPLE) epilogue_sample_tile<BN, AT, 4>(tmem_base, warp, lane, m0, n0, M, N, ep, tmem_full_bar, 0, -1);
    else epilogue_tile<BN, EPI, AT>(tmem_base, sA, sbias, warp, lane, m0, n0, M, N, ep, tmem_full_bar);
    tc_fence_before();
  }
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc(tmem_base, C::TMEM_COLS);
  }
#endif
}


// ------------------------------------------------------------------------------------------------
// tcgen05 / TMA GEMM on CTA pairs (cta_group::2).  A cluster of two CTAs computes a 256 x BN tile: CTA r stages
// rows [r*128, r*128+128) of A and rows [r*BN/2, (r+1)*BN/2) of the W tile; the leader's single MMA thread issues
// tcgen05.mma.cta_group::2 (M = 256, N = BN) which reads both CTAs' shared memory and accumulates rows r*128.. in CTA
// r's TMEM.  Per SM this halves the weight bytes staged per output row, which is what bounds these GEMMs: measured
// L2->SM ingest is ~84 GB/s per SM (profiles/r1_*), not the tensor pipe.
//   grid = (2 * N/BN, ceil(M/256)), cluster (2,1,1); warps 0 / 1 as in gemm_tc_kernel, warps 2-9 epilogue (two per
//   TMEM lane quarter, alternating 32-column chunks).
// tmA: [rows_pad, K] box {64,128}; tmW: [N, K] box {64, BN/2} (this CTA's half of the W tile, one load per stage); both
// SWIZZLE_128B.
// ------------------------------------------------------------------------------------------------
// KS = 64-wide k-blocks per ring stage.  The main loop of these GEMMs is NOT bound by bytes: a successful
// mbarrier.try_wait costs ~190-230 clk in the waiting thread and a TMA issue ~130 clk (+ ~64 per further instruction)
// whatever the box size (scripts/sm_ingest_bench.cu, profiles/r2_sm_ingest_bench.txt: 195 ns per iteration for 8, 16 or
// 32 KB boxes, ring depth 2..16, 1 or 144 CTAs), so with one k-block per stage the producer and the MMA issuer each
// spend ~300 ns per k-block on barrier round trips - the "78 GB/s per SM" of round 1 was that loop, not an ingest
// limit.  With KS = 2 one 3-D TMA box ([K/64][rows][64] view, box {64, rows, 2}) stages 128 columns of K per operand
// and the barrier waits / commits are paid once per 128 columns.  KS = 1 (2-D boxes) remains for K ranges with an odd
// number of k-blocks.
template <int BN, int KS = 1>
struct Tc2Cfg {
  static constexpr int BK = 64;
  static constexpr int A_ATOM = 128 * BK * 2;           // this CTA's 128 rows of A, one k-block
  static constexpr int B_ATOM = (BN / 2) * BK * 2;      // this CTA's half of the W tile, one k-block
  static constexpr int A_BYTES = KS * A_ATOM;
  static constexpr int B_BYTES = KS * B_ATOM;
  static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
  // >= 120 KB of shared memory per CTA on purpose: at most ONE GEMM CTA is resident per SM.  With two (the next
  // kernel's CTA launched early by PDL next to the current one) tcgen05.alloc/dealloc of different CTA pairs interleave
  // on the same SM pair, and the sampling loop was seen to hang in that state (round-1 notes, DESIGN.md 3.1).
  // One ring for both operands.  A second, deeper ring for the weight tiles with its own producer warp (requested up to
  // the whole K range ahead, before griddepcontrol.wait) was built and measured: no gain (3 198 vs 3 240 images/s) - with
  // the issue overhead gone these main loops run at the L2 -> SM throughput of the chip (~13-15 TB/s), not at DRAM latency.
  static constexpr int RING_BUDGET = KS == 1 ? 172032 : 196608;
  static constexpr int MAX_STAGES = KS == 1 ? 8 : 4;
  static constexpr int STAGES = (RING_BUDGET / STAGE_BYTES) > MAX_STAGES ? MAX_STAGES : (RING_BUDGET / STAGE_BYTES);
  static constexpr int ACC_COLS = BN <= 32 ? 32 : (BN <= 64 ? 64 : (BN <= 128 ? 128 : 256));   // one accumulator
  static constexpr int TMEM_COLS = 2 * ACC_COLS;                                               // double buffered
  static constexpr int EPI_WARPS = 8;                   // two per TMEM lane quarter
  static constexpr int THREADS = (2 + EPI_WARPS) * 32;
  static constexpr int SLAB_BYTES = EPI_WARPS * 4096;   // epilogue staging: one 32-row x 128 B slab per warp
  static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + SLAB_BYTES + 1024 /*align slack*/ + 256 /*barriers*/ + 1024 /*bias*/;
  static_assert(SMEM_BYTES <= 232448, "shared memory per CTA");
};

// arrive on the mbarrier at the same offset in CTA `cta` of the cluster
__device__ __forceinline__ void mbar_arrive_remote(uint64_t* bar, uint32_t cta) {
#if defined(__CUDA_ARCH__)
  uint32_t remote;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(remote) : "r"(smem_u32(bar)), "r"(cta));
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(remote) : "memory");
#endif
}

// Persistent over output tiles: grid.x = 2 * min(tiles, 74) CTAs; pair p computes tiles p, p + pairs, ...  The smem ring
// and its mbarrier phases run on across tiles, the accumulator is double buffered in TMEM (tile i+1's MMAs start while
// tile i is drained), so a GEMM with more tiles than pairs pays the fixed per-wave cost once.
// tile index -> (split z, row block, column block), column block fastest.
template <int BN, int EPI, typename AT, int KS = 1>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(Tc2Cfg<BN, KS>::THREADS, 1)
gemm_tc2_kernel(int trace_id, const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmW, int M,
                int N, int K, int w_row_off, int splits, EpiParams<AT> ep) {
#if defined(__CUDA_ARCH__)
  TraceScope trace_scope(trace_id);
  using C = Tc2Cfg<BN, KS>;
  static_assert(BN % 32 == 0 && BN >= 32 && BN <= 256, "pair tile width");
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~static_cast<uintptr_t>(1023));
  uint8_t* sA = smem;
  uint8_t* sB = smem + C::STAGES * C::A_BYTES;
  uint8_t* slab = sB + C::STAGES * C::B_BYTES;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(slab + C::SLAB_BYTES);
  uint64_t* empty_bar = full_bar + C::STAGES;
  uint64_t* tmem_full_bar = empty_bar + C::STAGES;       // [2]
  uint64_t* tmem_empty_bar = tmem_full_bar + 2;          // [2], used in the leader CTA only
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_empty_bar + 2);
  float* sbias = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(full_bar) + 256);

  const int warp = __shfl_sync(0xffffffffu, static_cast<int>(threadIdx.x >> 5), 0);   // provably warp-uniform (role dispatch)
  const int lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const bool leader = rank == 0;
  const int pair = blockIdx.x >> 1, npairs = gridDim.x >> 1;
  const int nt = N / BN, mt = (M + 255) / 256;
  const int total_tiles = nt * mt * splits;
  const int num_kb = (K / C::BK) / splits;               // 64-wide k-blocks per tile
  const int num_st = (num_kb + KS - 1) / KS;             // ring stages per tile (KS k-blocks each; the last may be short)

  // hq_debug_gemm_phases: per-CTA %globaltimer stamps of this launch (0 start, 1 prologue done, 2 dependency resolved,
  // 3 first stage landed, 4 last MMA issued, 5 accumulator complete, 6 epilogue done, 7 end)
#if defined(HQ_PHASE_STAMPS)
  const bool pm = trace_id >= 0 && trace_id == g_hq_phase_id;
#else
  constexpr bool pm = false;
#endif
  if (threadIdx.x == 0) phase_mark_if(pm, 0);
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmW);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < C::STAGES; ++s) {
      mbar_init(&full_bar[s], 1);     // leader: one arrive.expect_tx covering both CTAs' bytes
      mbar_init(&empty_bar[s], 1);    // one multicast tcgen05.commit per use
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(&tmem_full_bar[b], 1);    // one multicast tcgen05.commit per tile
      mbar_init(&tmem_empty_bar[b], 2 * C::EPI_WARPS);   // the epilogue warps of both CTAs
    }
    fence_barrier_init();
  }
  if (warp == 2) {
    tmem_alloc_2sm(tmem_slot, C::TMEM_COLS);
    tmem_relinquish_2sm();
  }
  tc_fence_before();
  __syncwarp();
  cluster_sync_all();                 // peer's barriers are initialised before anything signals them
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  if (threadIdx.x == 0) phase_mark_if(pm, 1);

  pdl_launch_dependents();
  if (warp == 0) {
    // ---- TMA producer (both CTAs; the whole warp runs the loop, one elected lane issues): own A rows + own half of
    //      the W tile, credited to the leader's full barrier.  The first ring of W tiles is requested before
    //      griddepcontrol.wait (weights never depend on the previous kernel), the activation tiles after it. ----
    int g = 0;                                          // ring stages issued so far (all tiles)
    bool first = true;
    for (int tile = pair; tile < total_tiles; tile += npairs) {
      const int z = tile / (nt * mt), rem = tile % (nt * mt);
      const int m0 = (rem / nt) * 256 + static_cast<int>(rank) * 128;
      const int wrow = w_row_off + (rem % nt) * BN + static_cast<int>(rank) * (BN / 2);
      const int kb0 = z * num_kb;
      // one instruction per operand and stage: KS = 1 a 2-D box of one k-block, KS > 1 a 3-D box of KS k-blocks
      // (a box that runs past this tile's K range lands whole - zero-filled past the matrix - and its surplus
      // k-blocks are simply not multiplied)
      auto load_a = [&](int st, int slot) {
        if (KS == 1) tma_load_2d_2sm(sA + slot * C::A_BYTES, &tmA, &full_bar[slot], (kb0 + st) * C::BK, m0);
        else tma_load_3d_2sm(sA + slot * C::A_BYTES, &tmA, &full_bar[slot], 0, m0, kb0 + st * KS);
      };
      auto load_w = [&](int st, int slot) {
        if (KS == 1) tma_load_2d_2sm(sB + slot * C::B_BYTES, &tmW, &full_bar[slot], (kb0 + st) * C::BK, wrow);
        else tma_load_3d_2sm(sB + slot * C::B_BYTES, &tmW, &full_bar[slot], 0, wrow, kb0 + st * KS);
      };
      int st = 0;
      if (first) {
        first = false;
        const int pre = num_st < C::STAGES ? num_st : C::STAGES;
        if (elect_one()) {
          for (int k2 = 0; k2 < pre; ++k2) {
            if (leader) mbar_arrive_expect_tx(&full_bar[k2], 2 * C::STAGE_BYTES);
            load_w(k2, k2);
          }
        }
        pdl_wait();
        if (lane == 0) phase_mark_if(pm, 2);
        if (elect_one()) {
          for (int k2 = 0; k2 < pre; ++k2) load_a(k2, k2);
        }
        st = pre;
        g = pre;
      }
      const bool prof = ep.prof != nullptr && blockIdx.x == 0;
      long long p_wait = 0, p_issue = 0, p_n = 0;
      const long long p_t0 = prof ? clock64() : 0;
      for (; st < num_st; ++st, ++g) {
        const int s = g % C::STAGES;
        const uint32_t ph = (g / C::STAGES) & 1;
        const long long c0 = prof ? clock64() : 0;
        mbar_wait(&empty_bar[s], ph ^ 1);
        const long long c1 = prof ? clock64() : 0;
        if (elect_one()) {
          if (leader) mbar_arrive_expect_tx(&full_bar[s], 2 * C::STAGE_BYTES);
          load_a(st, s);
          load_w(st, s);
        }
        if (prof) { p_wait += c1 - c0; p_issue += clock64() - c1; ++p_n; }
      }
      if (prof && lane == 0) { ep.prof[0] = p_wait; ep.prof[1] = p_issue; ep.prof[2] = clock64() - p_t0; ep.prof[3] = p_n; }
    }
  } else if (warp == 1) {
    if (leader) {
      // ---- MMA issuer (leader CTA only; warp-uniform loop, the elected lane issues the MMAs and their commits) ----
      constexpr uint32_t idesc = umma_idesc<AT>(256, BN);
      const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem_base, 0);
      int g = 0, it = 0;
      for (int tile = pair; tile < total_tiles; tile += npairs, ++it) {
        const int buf = it & 1;
        mbar_wait(&tmem_empty_bar[buf], ((it >> 1) & 1) ^ 1);     // both CTAs drained this accumulator
        tc_fence_after();
        const uint32_t acc = tmem_u + static_cast<uint32_t>(buf * C::ACC_COLS);
        const bool prof = ep.prof != nullptr && blockIdx.x == 0;
        long long m_wait = 0, m_issue = 0;
        const long long m_t0 = prof ? clock64() : 0;
        for (int st = 0; st < num_st; ++st, ++g) {
          const int s = g % C::STAGES;
          const uint32_t ph = (g / C::STAGES) & 1;
          const long long c0 = prof ? clock64() : 0;
          mbar_wait(&full_bar[s], ph);
          const long long c1 = prof ? clock64() : 0;
          if (g == 0 && lane == 0) phase_mark_if(pm, 3);
          tc_fence_after();
          if (elect_one()) {
#pragma unroll
            for (int j = 0; j < KS; ++j) {
              if (KS > 1 && st * KS + j >= num_kb) break;      // short last stage
              const uint64_t da = umma_smem_desc_sw128(smem_u32(sA + s * C::A_BYTES + j * C::A_ATOM));
              const uint64_t db = umma_smem_desc_sw128(smem_u32(sB + s * C::B_BYTES + j * C::B_ATOM));
#pragma unroll
              for (int k = 0; k < C::BK / 16; ++k)
                umma_bf16_2sm(acc, da + static_cast<uint64_t>(2 * k), db + static_cast<uint64_t>(2 * k), idesc,
                              (st > 0 || j > 0 || k > 0) ? 1u : 0u);
            }
            umma_commit_2sm(&empty_bar[s], 0x3);   // both CTAs may refill this slot
          }
          if (prof) { m_wait += c1 - c0; m_issue += clock64() - c1; }
        }
        if (prof && lane == 0) { ep.prof[4] = m_wait; ep.prof[5] = m_issue; ep.prof[6] = 0; ep.prof[7] = clock64() - m_t0; ep.prof[8] = num_st; }
        if (elect_one()) umma_commit_2sm(&tmem_full_bar[buf], 0x3);   // both CTAs' accumulators of this tile are complete
        if (lane == 0) phase_mark_if(pm, 4);
      }
    }
  } else {
    // ---- epilogue: this CTA's 128 rows of every tile (TMEM -> registers -> smem slab -> coalesced global) ----
    pdl_wait();
    int it = 0;
    for (int tile = pair; tile < total_tiles; tile += npairs, ++it) {
      const int buf = it & 1;
      const int z = tile / (nt * mt), rem = tile % (nt * mt);
      const int m0 = (rem / nt) * 256 + static_cast<int>(rank) * 128;
      const int n0 = (rem % nt) * BN;
      EpiParams<AT> ept = ep;
      if (EPI == EPI_F32) ept.outf = ep.outf + static_cast<size_t>(z) * ep.split_stride;
      if (EPI == EPI_SAMPLE)
        epilogue_sample_tile<BN, AT, C::EPI_WARPS>(tmem_base + static_cast<uint32_t>(buf * C::ACC_COLS), warp, lane, m0, n0, M, N,
                                                   ept, &tmem_full_bar[buf], (it >> 1) & 1, (warp & 3) + ((warp - 2) >> 2) * 4);
      else
        epilogue_tile<BN, EPI, AT, C::EPI_WARPS>(tmem_base + static_cast<uint32_t>(buf * C::ACC_COLS), slab, sbias, warp, lane, m0,
                                                 n0, M, N, ept, &tmem_full_bar[buf], (it >> 1) & 1,
                                                 (warp & 3) + ((warp - 2) >> 2) * 4, pm);
      tc_fence_before();
      __syncwarp();
      if (warp == 2 && lane == 0) phase_mark_if(pm, 6);
      // this warp is done with the accumulator (nobody waits for that after the pair's last tile: no remote signal then,
      // so that the tear-down barrier below needs no memory ordering)
      if (lane == 0 && tile + npairs < total_tiles) mbar_arrive_remote(&tmem_empty_bar[buf], 0);
    }
  }
  __syncwarp();
  // Both CTAs are done with each other's shared memory and TMEM before either frees them.  Execution barrier only: the
  // last cross-CTA signals (the leader's multicast commits) were consumed by the waits above; with the release form every
  // epilogue thread first waited here for its global stores to drain.
  cluster_sync_relaxed();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc_2sm(tmem_base, C::TMEM_COLS);
  }
  if (threadIdx.x == 0) phase_mark_if(pm, 7);
#endif
}

// ------------------------------------------------------------------------------------------------
// fp32 CUDA-core GEMM: 64 x 128 tile, BK = 16, 256 threads, 4 x 8 outputs per thread.
// A [M, K] and W [N, K] row-major fp32 (K % 16 == 0, N % 8 == 0).
// ------------------------------------------------------------------------------------------------
template <int EPI>
__global__ void __launch_bounds__(256)
gemm_simt_kernel(int trace_id, const float* __restrict__ A, const float* __restrict__ W, int M, int N, int K, EpiParams<float> ep) {
  constexpr int BM = 64, BN = 128, BK = 16;
  TraceScope trace_scope(trace_id);
  pdl_launch_dependents();
  pdl_wait();
  __shared__ __align__(16) float As[BK][BM + 4];
  __shared__ __align__(16) float Ws[BK][BN + 4];
  const int tid = threadIdx.x;
  const int tx = tid & 15;   // column group: cols tx*8 .. +8
  const int ty = tid >> 4;   // row group: rows ty*4 .. +4
  const int m0 = blockIdx.y * BM, n0 = blockIdx.x * BN;
  float acc[4][8];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;

  const int a_row = tid >> 2, a_k = (tid & 3) * 4;  // 64 rows x 4 float4
  for (int k0 = 0; k0 < K; k0 += BK) {
    {
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (m0 + a_row < M) v = *reinterpret_cast<const float4*>(A + static_cast<size_t>(m0 + a_row) * K + k0 + a_k);
      As[a_k + 0][a_row] = v.x; As[a_k + 1][a_row] = v.y; As[a_k + 2][a_row] = v.z; As[a_k + 3][a_row] = v.w;
    }
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int w_row = (tid >> 2) + h * 64;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (n0 + w_row < N) v = *reinterpret_cast<const float4*>(W + static_cast<size_t>(n0 + w_row) * K + k0 + a_k);
      Ws[a_k + 0][w_row] = v.x; Ws[a_k + 1][w_row] = v.y; Ws[a_k + 2][w_row] = v.z; Ws[a_k + 3][w_row] = v.w;
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < BK; ++k) {
      const float4 a = *reinterpret_cast<const float4*>(&As[k][ty * 4]);
      const float4 b0 = *reinterpret_cast<const float4*>(&Ws[k][tx * 8]);
      const float4 b1 = *reinterpret_cast<const float4*>(&Ws[k][tx * 8 + 4]);
      const float av[4] = {a.x, a.y, a.z, a.w};
      const float bv[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
    }
    __syncthreads();
  }
  const int n = n0 + tx * 8;
  if (n < N) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int m = m0 + ty * 4 + i;
      if (m < M) epi_store8<EPI, float>(ep, m, n, N, acc[i]);
    }
  }
}

}  // namespace hq
