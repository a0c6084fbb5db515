// Stage-1 decode of sampled code grids (SURVEY.md 8f-1): `SimRQGAN2Generator.decode_code`
// (hqvae/models/stage1/generator.py:312-367) for the shipped HQ-VAE configuration (decoding_type 'concat', upsample
// 'pixelshuffle'): codebook gather + PixelShuffle + concat -> post_quant_conv_b (1x1) -> VQGAN Decoder
// (stage1/modules/layers.py:300-410: conv_in, mid {ResnetBlock, AttnBlock, ResnetBlock}, per level {ResnetBlock (+ AttnBlock
// at the attention resolution)} x (num_res_blocks + 1) + nearest-2x Upsample conv, GroupNorm + swish + conv_out).
//
// Layout.  Activations are NHWC with a one-pixel ZERO border: a [B, H+2, W+2, C] tensor viewed as a matrix [B (H+2)(W+2), C].
// A 3x3 convolution is then nine SHIFTED GEMMs accumulated in TMEM: tap (ky, kx) reads the same matrix (ky-1)(W+2) + (kx-1)
// rows further down - one plain 2-D TMA tile load per k-block with a row offset, no im2col buffer, out-of-range rows are
// zero-filled by TMA - against the weight stored [Cout, 9 Cin] tap-major.  Outputs are computed for every padded position
// and the epilogue keeps only interior pixels, so borders stay zero.  The residual stream is fp32 (as in the sampler);
// GroupNorm (fp32 statistics, deterministic two-level reduction) writes the bf16 GEMM input.
//
// Operand type T.  The kernels that write or read convolution operands are templates over T:
//   bf16  (the default): kind::f16 MMAs; every convolution input and weight rounded to bf16 (nearest-even); q / k / v bf16.
//   float (precision tf32, what the reference computes: decode_code runs outside autocast and cuDNN runs its convolutions
//         in TF32): kind::tf32 MMAs with fp32 accumulation in TMEM.  Every convolution input - the codebook gather and its
//         PixelShuffle, the GroupNorm(+swish) output, the resample copy of x (nin_shortcut and upsample inputs), the
//         attention output (proj_out input) - and every conv weight is stored as fp32 rounded to TF32 with round-to-nearest,
//         ties away from zero (tf32_rna): the tensor core never sees low mantissa bits, so no result depends on how it treats
//         them.  The fused q | k | v convolution writes UNROUNDED fp32 and the AttnBlock core runs in fp32 on CUDA cores
//         (s1_attn_kernel<float>; PyTorch's default bmm does not use TF32).
// A 128-byte swizzled k-block row holds 64 bf16 or 32 fp32: the shared-memory geometry, stage bytes, swizzle and the
// descriptor advance per MMA (32 bytes: K = 16 bf16 or K = 8 tf32) are the same for both.
#pragma once

#include "chain.cuh"

namespace hq {

// fp32 -> TF32 (sign, 8-bit exponent, 10-bit mantissa) with round-to-nearest, ties away from zero; the low 13 bits are
// cleared whatever the conversion leaves in them.
__device__ __forceinline__ float tf32_rna(float v) {
  uint32_t u;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(u) : "f"(v));
  return __uint_as_float(u & 0xffffe000u);
}

// One fp32 value as a convolution operand of type T (bf16: nearest-even; float: TF32, ties away)
template <typename T> __device__ __forceinline__ T s1_round(float v);
template <> __device__ __forceinline__ bf16 s1_round<bf16>(float v) { return __float2bfloat16_rn(v); }
template <> __device__ __forceinline__ float s1_round<float>(float v) { return tf32_rna(v); }

// ------------------------------------------------------------------------------------------------
// implicit-GEMM convolution on CTA pairs (tcgen05, cta_group::2): 256 padded positions x bn output channels per tile
// ------------------------------------------------------------------------------------------------
// S1_OUT_ACT: a T matrix - bf16 rounded to nearest-even, or UNROUNDED fp32 in the tf32 instantiation (its one user, the
// q | k | v convolution, feeds the fp32 attention core)
enum { S1_OUT_F32 = 0, S1_OUT_ACT = 1, S1_OUT_IMAGE = 2 };

struct ConvParams {
  int R;            // padded positions in total (B * Hp * Wp) = rows of the A matrix
  int Cin, CoutPad, cout;   // CoutPad: weight rows (multiple of bn, zero-padded); cout: real output channels
  int taps;         // 1 (1x1) | 9 (3x3, padding 1)
  int Hp, Wp;       // padded height / width (H + 2, W + 2)
  int bn;           // tile width
  int mode;         // S1_OUT_*
  int ldo;          // row stride (elements) of the output matrix (modes 0 / 1)
  const float* bias;    // [CoutPad]
  const float* res;     // optional fp32 residual [R, ldo] (mode 0), may alias outf
  float* outf;          // mode 0: fp32 [R, ldo]; mode 2: image [B, cout, H, W] fp32
  void* outb;           // mode 1: T [R, ldo]
};

// T = bf16 (kind::f16) or float (kind::tf32; operands already rounded to TF32)
template <typename T>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(CH_THREADS, 1)
conv_tc2_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmW, ConvParams p) {
#if defined(__CUDA_ARCH__)
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~static_cast<uintptr_t>(1023));
  uint8_t* slab = smem + CH_STAGES * CH_STAGE_BYTES;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(slab + CH_SLAB_BYTES);
  uint64_t* empty_bar = full_bar + CH_STAGES;
  uint64_t* tmem_full_bar = empty_bar + CH_STAGES;
  uint64_t* tmem_empty_bar = tmem_full_bar + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_empty_bar + 2);
  float* sbias = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(full_bar) + 256);

  const int warp = __shfl_sync(0xffffffffu, static_cast<int>(threadIdx.x >> 5), 0);   // provably warp-uniform (role dispatch)
  const int lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const bool leader = rank == 0;
  const int pair = blockIdx.x >> 1, npairs = gridDim.x >> 1;
  const int bn = p.bn;
  const int nt = p.CoutPad / bn, mt = (p.R + 255) / 256;
  const int total_tiles = nt * mt;
  constexpr int KB = 128 / static_cast<int>(sizeof(T));   // elements per 128-byte k-block row
  const int kpt = p.Cin / KB;                       // k-blocks per tap
  const int num_kb = p.taps * kpt;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmW);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < CH_STAGES; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(&tmem_full_bar[b], 1);
      mbar_init(&tmem_empty_bar[b], 2 * CH_EPI_WARPS);
    }
    fence_barrier_init();
  }
  if (warp == 2) {
    tmem_alloc_2sm(tmem_slot, 2 * CH_ACC_COLS);
    tmem_relinquish_2sm();
  }
  tc_fence_before();
  __syncwarp();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ---- TMA producer (warp-uniform loop, one elected lane issues: see elect_one in common.cuh): tap (ky, kx) of a 3x3
    //      kernel reads the activation matrix (ky-1) Wp + (kx-1) rows below the output row; rows outside [0, R) are
    //      zero-filled by TMA.  Column tile fastest: the pairs working on the same row block at the same time share its
    //      A tiles through L2. ----
    const uint32_t stage_tx = 2u * static_cast<uint32_t>(CH_A_BYTES + bn * 64);
    uint32_t g = 0;
    for (int tile = pair; tile < total_tiles; tile += npairs) {
      const int m0 = (tile / nt) * 256 + static_cast<int>(rank) * 128;
      const int wrow = (tile % nt) * bn + static_cast<int>(rank) * (bn / 2);
      for (int kb = 0; kb < num_kb; ++kb, ++g) {
        const int tap = kb / kpt, kc = kb - tap * kpt;
        const int off = p.taps == 9 ? (tap / 3 - 1) * p.Wp + (tap % 3 - 1) : 0;
        const int s = static_cast<int>(g % CH_STAGES);
        mbar_wait(&empty_bar[s], ((g / CH_STAGES) & 1) ^ 1);
        if (elect_one()) {
          if (leader) mbar_arrive_expect_tx(&full_bar[s], stage_tx);
          tma_load_2d_2sm(smem + s * CH_STAGE_BYTES, &tmA, &full_bar[s], kc * KB, m0 + off);
          tma_load_2d_2sm(smem + s * CH_STAGE_BYTES + CH_A_BYTES, &tmW, &full_bar[s], kb * KB, wrow);
        }
      }
    }
  } else if (warp == 1) {
    if (leader) {
      // ---- MMA issuer (warp-uniform loop, the elected lane issues the MMAs and their commits) ----
      const uint32_t idesc = std::is_same<T, float>::value ? umma_idesc_tf32(256, bn) : umma_idesc_bf16(256, bn);
      const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem_base, 0);
      uint32_t g = 0, it = 0;
      for (int tile = pair; tile < total_tiles; tile += npairs, ++it) {
        const uint32_t buf = it & 1;
        mbar_wait(&tmem_empty_bar[buf], ((it >> 1) & 1) ^ 1);
        tc_fence_after();
        const uint32_t acc = tmem_u + buf * CH_ACC_COLS;
        for (int kb = 0; kb < num_kb; ++kb, ++g) {
          const int s = static_cast<int>(g % CH_STAGES);
          mbar_wait(&full_bar[s], (g / CH_STAGES) & 1);
          tc_fence_after();
          if (elect_one()) {
            const uint64_t da = umma_smem_desc_sw128(smem_u32(smem + s * CH_STAGE_BYTES));
            const uint64_t db = umma_smem_desc_sw128(smem_u32(smem + s * CH_STAGE_BYTES + CH_A_BYTES));
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              if constexpr (std::is_same<T, float>::value)
                umma_tf32_2sm(acc, da + static_cast<uint64_t>(2 * k), db + static_cast<uint64_t>(2 * k), idesc,
                              (kb > 0 || k > 0) ? 1u : 0u);
              else
                umma_bf16_2sm(acc, da + static_cast<uint64_t>(2 * k), db + static_cast<uint64_t>(2 * k), idesc,
                              (kb > 0 || k > 0) ? 1u : 0u);
            }
            umma_commit_2sm(&empty_bar[s], 0x3);
          }
        }
        if (elect_one()) umma_commit_2sm(&tmem_full_bar[buf], 0x3);
      }
    }
  } else {
    // ---- epilogue: bias (+ fp32 residual), interior pixels only ----
    const int ew = (warp & 3) + ((warp - 2) >> 2) * 4;
    const int quarter = warp & 3, half = ew >> 2;
    const int etid = ew * 32 + lane;
    const int piece = lane & 7;
    const int HpWp = p.Hp * p.Wp, H = p.Hp - 2, W = p.Wp - 2;
    uint8_t* myslab = slab + ew * 4096;
    const uint32_t slab_u32 = smem_u32(myslab);
    uint32_t it = 0;
    for (int tile = pair; tile < total_tiles; tile += npairs, ++it) {
      const uint32_t buf = it & 1;
      const int m0 = (tile / nt) * 256 + static_cast<int>(rank) * 128;
      const int n0 = (tile % nt) * bn;
      named_bar(1, 256);
      for (int i = etid; i < bn; i += 256) sbias[i] = p.bias[n0 + i];
      // rows this lane writes: it8*4 + (lane >> 3) of the warp's 32
      bool row_ok[8];
      size_t row_off[8];
#pragma unroll
      for (int r8 = 0; r8 < 8; ++r8) {
        const int m = m0 + quarter * 32 + r8 * 4 + (lane >> 3);
        const int b = m / HpWp, q = m - b * HpWp;
        const int y = q / p.Wp, x = q - y * p.Wp;
        row_ok[r8] = m < p.R && y >= 1 && y <= H && x >= 1 && x <= W;
        row_off[r8] = p.mode == S1_OUT_IMAGE ? (static_cast<size_t>(b) * p.cout * H + (y - 1)) * W + (x - 1)
                                             : static_cast<size_t>(m) * p.ldo;
      }
      named_bar(1, 256);
      mbar_wait(&tmem_full_bar[buf], (it >> 1) & 1);
      tc_fence_after();
      const uint32_t acc = tmem_base + buf * CH_ACC_COLS;
#pragma unroll 1
      for (int c = half; c < bn / 32; c += 2) {
        // residual of this lane's 8 rows x 4 columns: requested before the TMEM load so that its latency hides behind
        // the transposition (ncu: the layers with a residual were ~120 us slower than their twins without one)
        float4 resid[8];
        const int colp = n0 + c * 32 + piece * 4;
        if (p.mode == S1_OUT_F32 && p.res != nullptr && colp < p.cout) {
#pragma unroll
          for (int r8 = 0; r8 < 8; ++r8)
            resid[r8] = row_ok[r8] ? *reinterpret_cast<const float4*>(p.res + row_off[r8] + colp) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
        uint32_t r[32];
        tmem_ld_32x32(acc + (static_cast<uint32_t>(quarter * 32) << 16) + static_cast<uint32_t>(c * 32), r);
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const uint32_t addr = slab_u32 + lane * 128 + ((j ^ (lane & 7)) << 4);
          asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(r[4 * j]), "r"(r[4 * j + 1]),
                       "r"(r[4 * j + 2]), "r"(r[4 * j + 3])
                       : "memory");
        }
        __syncwarp();
        const int col = n0 + c * 32 + piece * 4;
        const float4 b4 = *reinterpret_cast<const float4*>(sbias + c * 32 + piece * 4);
        if (col < p.cout) {
#pragma unroll
          for (int r8 = 0; r8 < 8; ++r8) {
            const int row = r8 * 4 + (lane >> 3);
            float4 v;
            const uint32_t addr = slab_u32 + row * 128 + ((piece ^ (row & 7)) << 4);
            asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
            v.x += b4.x; v.y += b4.y; v.z += b4.z; v.w += b4.w;
            if (!row_ok[r8]) continue;
            if (p.mode == S1_OUT_F32) {
              float4* dst = reinterpret_cast<float4*>(p.outf + row_off[r8] + col);
              if (p.res != nullptr) {
                const float4 a = resid[r8];
                v.x += a.x; v.y += a.y; v.z += a.z; v.w += a.w;
              }
              *dst = v;
            } else if (p.mode == S1_OUT_ACT) {
              if constexpr (std::is_same<T, float>::value) {
                *reinterpret_cast<float4*>(static_cast<float*>(p.outb) + row_off[r8] + col) = v;
              } else {
                uint2 u;
                __nv_bfloat162 h0 = __floats2bfloat162_rn(v.x, v.y), h1 = __floats2bfloat162_rn(v.z, v.w);
                u.x = *reinterpret_cast<uint32_t*>(&h0);
                u.y = *reinterpret_cast<uint32_t*>(&h1);
                *reinterpret_cast<uint2*>(static_cast<bf16*>(p.outb) + row_off[r8] + col) = u;
              }
            } else {
              const float vv[4] = {v.x, v.y, v.z, v.w};
              const size_t plane = static_cast<size_t>(H) * W;
#pragma unroll
              for (int e = 0; e < 4; ++e)
                if (col + e < p.cout) p.outf[row_off[r8] + static_cast<size_t>(col + e) * plane] = vv[e];
            }
          }
        }
        __syncwarp();
      }
      tc_fence_before();
      __syncwarp();
      // no remote signal after the pair's last tile (nobody waits for it): the tear-down barrier below then needs no
      // memory ordering, and the epilogue threads do not wait there for their global stores to drain (see gemm_tc2_kernel)
      if (lane == 0 && tile + npairs < total_tiles) mbar_arrive_remote(&tmem_empty_bar[buf], 0);
    }
  }
  __syncwarp();
  cluster_sync_relaxed();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc_2sm(tmem_base, 2 * CH_ACC_COLS);
  }
#endif
}

// ------------------------------------------------------------------------------------------------
// element-wise / reduction kernels of the decoder
// ------------------------------------------------------------------------------------------------
// codes -> input of post_quant_conv_b (generator.py:316-319): channels [0, E) = PixelShuffle(2) of the top entry (E*4 wide:
// out[c, y, x] = in[4c + 2 (y % 2) + (x % 2), y / 2, x / 2]), channels [E, 2E) = the bottom entry.  One CTA per bottom pixel.
template <typename T>
__global__ void __launch_bounds__(256)
s1_quant_kernel(const int64_t* __restrict__ code_t, const int64_t* __restrict__ code_b, const float* __restrict__ E_t,
                const float* __restrict__ E_b, T* __restrict__ out, int E, int hb /*bottom grid side*/, int n_embed) {
  const int Wp = hb + 2;
  const int pp = blockIdx.x;                   // padded pixel: b * Wp * Wp + yp * Wp + xp
  const int b = pp / (Wp * Wp), q = pp % (Wp * Wp), y = q / Wp - 1, x = q % Wp - 1;
  T* o = out + static_cast<size_t>(pp) * 2 * E;
  const int ht = hb / 2;
  int64_t ct = -1, cb = -1;
  if (y >= 0 && y < hb && x >= 0 && x < hb) {
    ct = code_t[(static_cast<size_t>(b) * ht + y / 2) * ht + x / 2];
    cb = code_b[(static_cast<size_t>(b) * hb + y) * hb + x];
  }
  if (ct < 0 || ct >= n_embed || cb < 0 || cb >= n_embed) {      // border (or an out-of-range code: the host validates)
    for (int c = threadIdx.x; c < 2 * E; c += blockDim.x) o[c] = s1_round<T>(0.f);
    return;
  }
  const float* et = E_t + static_cast<size_t>(ct) * 4 * E + 2 * (y & 1) + (x & 1);
  const float* eb = E_b + static_cast<size_t>(cb) * E;
  for (int c = threadIdx.x; c < E; c += blockDim.x) {
    o[c] = s1_round<T>(et[4 * c]);
    o[E + c] = s1_round<T>(eb[c]);
  }
}

// GroupNorm(32 groups, eps 1e-6; layers.py:17-21) statistics over the interior of a padded fp32 NHWC tensor: partial (sum,
// sum of squares) per (image, group, slice of rows); grid (S slices, B).  Every element is read once, as float4 along the
// channels (thread = channel quad x pixel lane, four loads in flight per thread); threads keep fp32 partials of <= a few
// hundred terms, the cross-thread reduction runs in double in a FIXED order, and the LAST slice CTA of an image to finish
// (ticket counter that wraps back to 0) adds the S slices in a fixed order and publishes (mean, rstd) per group: the
// result does not depend on which CTA happens to be last.
__global__ void __launch_bounds__(256)
s1_gn_stats_kernel(const float* __restrict__ x, double* __restrict__ part, float2* __restrict__ stat, unsigned* __restrict__ cnt,
                   int Hp, int Wp, int C, int S) {
  const int s = blockIdx.x, b = blockIdx.y;
  const int H = Hp - 2, W = Wp - 2, c4 = C / 4, cg = C / 32;
  const int P = 256 / c4 > 0 ? 256 / c4 : 1;           // pixel lanes (C <= 1024)
  const int tid = threadIdx.x, q = tid % c4, pl = tid / c4;
  const int rows_per = (H + S - 1) / S;
  const int y0 = s * rows_per, y1 = min(H, y0 + rows_per);
  const int npx = (y1 - y0) * W;
  float4 sum = make_float4(0.f, 0.f, 0.f, 0.f), sq = make_float4(0.f, 0.f, 0.f, 0.f);
  if (pl < P && tid < c4 * P) {
    const float* xb = x + (static_cast<size_t>(b) * Hp * Wp) * C + 4 * q;
    auto at = [&](int i) { return xb + (static_cast<size_t>(y0 + i / W + 1) * Wp + i % W + 1) * C; };
    int i = pl;
    for (; i + 3 * P < npx; i += 4 * P) {
      const float4 v0 = *reinterpret_cast<const float4*>(at(i)), v1 = *reinterpret_cast<const float4*>(at(i + P));
      const float4 v2 = *reinterpret_cast<const float4*>(at(i + 2 * P)), v3 = *reinterpret_cast<const float4*>(at(i + 3 * P));
#define S1_ACC(v) sum.x += v.x; sum.y += v.y; sum.z += v.z; sum.w += v.w; \
  sq.x = fmaf(v.x, v.x, sq.x); sq.y = fmaf(v.y, v.y, sq.y); sq.z = fmaf(v.z, v.z, sq.z); sq.w = fmaf(v.w, v.w, sq.w);
      S1_ACC(v0) S1_ACC(v1) S1_ACC(v2) S1_ACC(v3)
    }
    for (; i < npx; i += P) {
      const float4 v = *reinterpret_cast<const float4*>(at(i));
      S1_ACC(v)
    }
#undef S1_ACC
  }
  __shared__ double ssum[256 * 4], ssq[256 * 4];
  __shared__ unsigned s_ticket;
  ssum[tid * 4 + 0] = sum.x; ssum[tid * 4 + 1] = sum.y; ssum[tid * 4 + 2] = sum.z; ssum[tid * 4 + 3] = sum.w;
  ssq[tid * 4 + 0] = sq.x; ssq[tid * 4 + 1] = sq.y; ssq[tid * 4 + 2] = sq.z; ssq[tid * 4 + 3] = sq.w;
  __syncthreads();
  if (tid < 32) {
    double a = 0.0, qq = 0.0;
    for (int p2 = 0; p2 < P; ++p2)
      for (int c = tid * cg; c < (tid + 1) * cg; ++c) {
        const int e = (p2 * c4 + c / 4) * 4 + (c & 3);
        a += ssum[e];
        qq += ssq[e];
      }
    double* o = part + ((static_cast<size_t>(b) * 32 + tid) * S + s) * 2;
    o[0] = a;
    o[1] = qq;
    __threadfence();
  }
  __syncthreads();
  if (tid == 0) s_ticket = atomicInc(cnt + b, static_cast<unsigned>(S - 1));
  __syncthreads();
  if (s_ticket == static_cast<unsigned>(S - 1) && tid < 32) {
    __threadfence();
    const double* pp = part + (static_cast<size_t>(b) * 32 + tid) * S * 2;
    double a = 0.0, qq = 0.0;
    for (int k = 0; k < S; ++k) { a += __ldcg(pp + 2 * k); qq += __ldcg(pp + 2 * k + 1); }
    const double n = static_cast<double>(H) * W * cg;
    const double mean = a / n;
    double var = qq / n - mean * mean;
    if (var < 0.0) var = 0.0;
    stat[b * 32 + tid] = make_float2(static_cast<float>(mean), static_cast<float>(1.0 / sqrt(var + 1e-6)));
  }
}

// x * sigmoid(x) (layers.py:12-14) with the fast exponential / division: ~1e-6 relative, far below the bf16 rounding of the output
__device__ __forceinline__ float swish_f(float v) { return __fdividef(v, 1.0f + __expf(-v)); }

// y = GroupNorm(x) (optionally * sigmoid) as T; EVERY padded position is written, the border with zeros (the buffers are
// reused at other resolutions: a 3x3 convolution must find zeros around its input).  One CTA per padded row (b, y), four
// float4 loads in flight per thread.
template <typename T>
__global__ void __launch_bounds__(256)
s1_gn_apply_kernel(const float* __restrict__ x, const float2* __restrict__ stat, const float* __restrict__ gamma,
                   const float* __restrict__ beta, T* __restrict__ out, int Hp, int Wp, int C, int swish) {
  const int b = blockIdx.y, y = blockIdx.x;
  const int H = Hp - 2, W = Wp - 2, cg = C / 32;
  __shared__ float s_mean[32], s_rstd[32];
  if (threadIdx.x < 32) {
    const float2 st = stat[b * 32 + threadIdx.x];
    s_mean[threadIdx.x] = st.x;
    s_rstd[threadIdx.x] = st.y;
  }
  __syncthreads();
  const int c4 = C / 4, total = Wp * c4;
  const size_t base = (static_cast<size_t>(b) * Hp + y) * Wp * C;
  const bool row_in = y >= 1 && y <= H;
  for (int i0 = threadIdx.x; i0 < total; i0 += 4 * 256) {
    float4 v[4];
    int off[4];
    bool in[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const int i = i0 + k * 256, xx = i / c4;
      off[k] = i < total ? xx * C + (i - xx * c4) * 4 : -1;
      in[k] = i < total && row_in && xx >= 1 && xx <= W;
      if (in[k]) v[k] = *reinterpret_cast<const float4*>(x + base + off[k]);
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      if (off[k] < 0) continue;
      uint2 u = make_uint2(0u, 0u);
      float4 f = make_float4(0.f, 0.f, 0.f, 0.f);
      if (in[k]) {
        const int c = (i0 + k * 256) % c4 * 4;
        const float4 ga = *reinterpret_cast<const float4*>(gamma + c);
        const float4 be = *reinterpret_cast<const float4*>(beta + c);
        int g0 = c / cg, g1 = g0, g2 = g0, g3 = g0;
        if (cg & 3) { g1 = (c + 1) / cg; g2 = (c + 2) / cg; g3 = (c + 3) / cg; }
        float o0 = (v[k].x - s_mean[g0]) * s_rstd[g0] * ga.x + be.x, o1 = (v[k].y - s_mean[g1]) * s_rstd[g1] * ga.y + be.y;
        float o2 = (v[k].z - s_mean[g2]) * s_rstd[g2] * ga.z + be.z, o3 = (v[k].w - s_mean[g3]) * s_rstd[g3] * ga.w + be.w;
        if (swish) { o0 = swish_f(o0); o1 = swish_f(o1); o2 = swish_f(o2); o3 = swish_f(o3); }
        if constexpr (std::is_same<T, float>::value) {
          f = make_float4(tf32_rna(o0), tf32_rna(o1), tf32_rna(o2), tf32_rna(o3));
        } else {
          __nv_bfloat162 h0 = __floats2bfloat162_rn(o0, o1), h1 = __floats2bfloat162_rn(o2, o3);
          u.x = *reinterpret_cast<uint32_t*>(&h0);
          u.y = *reinterpret_cast<uint32_t*>(&h1);
        }
      }
      if constexpr (std::is_same<T, float>::value) *reinterpret_cast<float4*>(out + base + off[k]) = f;
      else *reinterpret_cast<uint2*>(out + base + off[k]) = u;
    }
  }
}

// nearest-neighbour 2x upsampling (Upsample, layers.py:49-52) fp32 [B, H+2, W+2, C] -> T [B, 2H+2, 2W+2, C]: the input
// of the level's upsample convolution.  up = 1: plain fp32 -> T copy of the interior (input of a nin_shortcut 1x1 conv).
template <typename T>
__global__ void __launch_bounds__(256)
s1_resample_kernel(const float* __restrict__ x, T* __restrict__ out, int H, int W, int C, int up) {
  const int b = blockIdx.y, yp = blockIdx.x;           // output padded row 0 .. up*H+1
  const int Ho = up * H, Wo = up * W, c4 = C / 4;
  T* dst = out + ((static_cast<size_t>(b) * (Ho + 2) + yp) * (Wo + 2)) * C;
  const bool row_in = yp >= 1 && yp <= Ho;
  const float* src = x + ((static_cast<size_t>(b) * (H + 2) + (row_in ? (yp - 1) / up + 1 : 0)) * (W + 2)) * C;
  for (int i = threadIdx.x; i < (Wo + 2) * c4; i += blockDim.x) {
    const int xp = i / c4, c = (i % c4) * 4;
    uint2 u = make_uint2(0u, 0u);
    float4 f = make_float4(0.f, 0.f, 0.f, 0.f);
    if (row_in && xp >= 1 && xp <= Wo) {
      const float4 v = *reinterpret_cast<const float4*>(src + static_cast<size_t>((xp - 1) / up + 1) * C + c);
      if constexpr (std::is_same<T, float>::value) {
        f = make_float4(tf32_rna(v.x), tf32_rna(v.y), tf32_rna(v.z), tf32_rna(v.w));
      } else {
        __nv_bfloat162 h0 = __floats2bfloat162_rn(v.x, v.y), h1 = __floats2bfloat162_rn(v.z, v.w);
        u.x = *reinterpret_cast<uint32_t*>(&h0);
        u.y = *reinterpret_cast<uint32_t*>(&h1);
      }
    }
    if constexpr (std::is_same<T, float>::value) *reinterpret_cast<float4*>(dst + static_cast<size_t>(xp) * C + c) = f;
    else *reinterpret_cast<uint2*>(dst + static_cast<size_t>(xp) * C + c) = u;
  }
}

// AttnBlock core (layers.py:170-183): single-head attention over the N = H W pixels of an image, C channels, scale C^-1/2.
// qkv: T padded [B, Hp, Wp, 3C] (q | k | v along channels); out: T padded [B, Hp, Wp, C] (interior only), a proj_out input
// (s1_round).  One CTA (256 threads) per (image, tile of S1_ATT_Q queries): scores in shared memory, full softmax, then P V.
constexpr int S1_ATT_Q = 8;
template <typename T>
__global__ void __launch_bounds__(256)
s1_attn_kernel(const T* __restrict__ qkv, T* __restrict__ out, int H, int W, int C) {
  extern __shared__ float s1_att_smem[];
  const int N = H * W, Wp = W + 2;
  float* sq = s1_att_smem;                     // [S1_ATT_Q][C]
  float* sp = sq + S1_ATT_Q * C;               // [S1_ATT_Q][N]
  __shared__ float red[S1_ATT_Q][8];
  const int b = blockIdx.y, q0 = blockIdx.x * S1_ATT_Q;
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const size_t img = static_cast<size_t>(b) * (H + 2) * Wp;
  auto prow = [&](int n) { return img + static_cast<size_t>(n / W + 1) * Wp + (n % W + 1); };
  for (int i = tid; i < S1_ATT_Q * C; i += blockDim.x) {
    const int qi = i / C, c = i % C, n = q0 + qi;
    sq[i] = n < N ? ActT<T>::to_f(qkv[prow(n) * 3 * C + c]) : 0.f;
  }
  __syncthreads();
  const float scale = rsqrtf(static_cast<float>(C));
  for (int j = tid; j < N; j += blockDim.x) {
    const T* kr = qkv + prow(j) * 3 * C + C;
    float acc[S1_ATT_Q];
#pragma unroll
    for (int qi = 0; qi < S1_ATT_Q; ++qi) acc[qi] = 0.f;
    for (int c = 0; c < C; c += 8) {
      float kv[8];
      load8(kr + c, kv);
#pragma unroll
      for (int qi = 0; qi < S1_ATT_Q; ++qi)
#pragma unroll
        for (int e = 0; e < 8; ++e) acc[qi] = fmaf(sq[qi * C + c + e], kv[e], acc[qi]);
    }
#pragma unroll
    for (int qi = 0; qi < S1_ATT_Q; ++qi) sp[qi * N + j] = acc[qi] * scale;
  }
  __syncthreads();
  // softmax over the keys of each query: warp `wid` owns query `wid`
  if (wid < S1_ATT_Q) {
    float mx = -INFINITY;
    for (int j = lane; j < N; j += 32) mx = fmaxf(mx, sp[wid * N + j]);
    mx = warp_max(mx);
    float sum = 0.f;
    for (int j = lane; j < N; j += 32) {
      const float e = expf(sp[wid * N + j] - mx);
      sp[wid * N + j] = e;
      sum += e;
    }
    sum = warp_sum(sum);
    if (lane == 0) red[wid][0] = 1.0f / sum;
  }
  __syncthreads();
  for (int c = tid * 2; c < C; c += blockDim.x * 2) {
    float a0[S1_ATT_Q], a1[S1_ATT_Q];
#pragma unroll
    for (int qi = 0; qi < S1_ATT_Q; ++qi) a0[qi] = a1[qi] = 0.f;
    for (int j = 0; j < N; ++j) {
      float2 vf;
      if constexpr (std::is_same<T, float>::value) {
        vf = *reinterpret_cast<const float2*>(qkv + prow(j) * 3 * C + 2 * C + c);
      } else {
        const __nv_bfloat162 v2 = *reinterpret_cast<const __nv_bfloat162*>(qkv + prow(j) * 3 * C + 2 * C + c);
        vf = __bfloat1622float2(v2);
      }
#pragma unroll
      for (int qi = 0; qi < S1_ATT_Q; ++qi) {
        const float w = sp[qi * N + j];
        a0[qi] = fmaf(w, vf.x, a0[qi]);
        a1[qi] = fmaf(w, vf.y, a1[qi]);
      }
    }
#pragma unroll
    for (int qi = 0; qi < S1_ATT_Q; ++qi) {
      const int n = q0 + qi;
      if (n < N) {
        const float inv = red[qi][0];
        if constexpr (std::is_same<T, float>::value)
          *reinterpret_cast<float2*>(out + prow(n) * C + c) = make_float2(tf32_rna(a0[qi] * inv), tf32_rna(a1[qi] * inv));
        else
          *reinterpret_cast<__nv_bfloat162*>(out + prow(n) * C + c) = __floats2bfloat162_rn(a0[qi] * inv, a1[qi] * inv);
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------
// AttnBlock core on the tensor cores (mma.sync m16n8k16 bf16, fp32 accumulate): the CUDA-core kernel above needs ~410 us per
// call at B = 32 (16 % of a decode); this one keeps a 64-query tile's scores in registers.
//   CTA = (image, 64 queries), 4 warps x 16 queries.  Phase 1: S = Q K^T over 64-key chunks of K staged in shared memory
//   (A = Q rows via ldmatrix.x4, B = K rows [key][channel] via ldmatrix.x2), softmax in registers (quad shuffles), P -> shared
//   memory as bf16.  Phase 2: O = P V per 128-channel block over 64-key tiles of V (B = V^T via ldmatrix.x2.trans).
//   N = H W <= 256 tokens (multiple of 16), C <= 512 channels (multiple of 64).
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void ldsm_x4(uint32_t addr, uint32_t& r0, uint32_t& r1, uint32_t& r2, uint32_t& r3) {
#if defined(__CUDA_ARCH__)
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];" : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3) : "r"(addr));
#endif
}
__device__ __forceinline__ void cp_async16(uint32_t dst, const void* src) {
#if defined(__CUDA_ARCH__)
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
#endif
}
__device__ __forceinline__ void cp_async_commit() {
#if defined(__CUDA_ARCH__)
  asm volatile("cp.async.commit_group;" ::: "memory");
#endif
}
template <int N>
__device__ __forceinline__ void cp_async_wait() {
#if defined(__CUDA_ARCH__)
  asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory");
#endif
}
// S1A_KC keys per K chunk (phase 1, ring of S1A_NKB buffers), S1A_VC keys x S1A_CB channels per V tile (phase 2, ring of
// S1A_NVB): cp.async prefetch S1A_NKB - 1 / S1A_NVB - 1 tiles ahead (one warp per scheduler: nothing else hides the latency)
constexpr int S1A_Q = 64, S1A_KC = 32, S1A_VC = 64, S1A_CB = 128, S1A_NMAX = 256, S1A_CMAX = 512, S1A_PAD = 8;
constexpr int S1A_NKB = 3, S1A_NVB = 4;
__host__ __device__ constexpr int s1a_kv_elems(int C) {
  return S1A_NKB * S1A_KC * (C + S1A_PAD) > S1A_NVB * S1A_VC * (S1A_CB + S1A_PAD) ? S1A_NKB * S1A_KC * (C + S1A_PAD)
                                                                                  : S1A_NVB * S1A_VC * (S1A_CB + S1A_PAD);
}
__host__ __device__ constexpr int s1a_smem_bytes(int C) {
  return (S1A_Q * (C + S1A_PAD) + s1a_kv_elems(C) + S1A_Q * (S1A_NMAX + S1A_PAD)) * 2;
}

__global__ void __launch_bounds__(128, 1)
s1_attn_mma_kernel(const bf16* __restrict__ qkv, bf16* __restrict__ out, int H, int W, int C) {
#if defined(__CUDA_ARCH__)
  extern __shared__ __align__(16) uint8_t s1a_smem[];
  const int N = H * W, Wp = W + 2;
  const int qp = C + S1A_PAD, pp = S1A_NMAX + S1A_PAD, vp = S1A_CB + S1A_PAD;      // row pitches (elements)
  bf16* Qs = reinterpret_cast<bf16*>(s1a_smem);                 // [64][C + 8]
  bf16* KV = Qs + S1A_Q * qp;                                   // 2 x K chunk [32][C + 8]; phase 2: 2 x V tile [64][128 + 8]
  bf16* Ps = KV + s1a_kv_elems(C);                              // [64][256 + 8]
  const int kbuf = S1A_KC * qp, vbuf = S1A_VC * vp;
  const int b = blockIdx.y, q0 = blockIdx.x * S1A_Q;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, t = lane & 3;
  const size_t img = static_cast<size_t>(b) * (H + 2) * Wp;
  __shared__ int tok[S1A_NMAX];                                 // padded-matrix row of token n (relative to the image)
  for (int n = tid; n < N; n += 128) tok[n] = (n / W + 1) * Wp + (n % W + 1);
  __syncthreads();
  auto prow = [&](int n) { return img + static_cast<size_t>(tok[n]); };
  const int c8 = C / 8;
  // tile loaders: 16-byte cp.async per thread, rows beyond N zero-filled; a thread keeps its column and walks the rows
  // (128 % ncol8 == 0 for C = 128 / 256 / 512; otherwise the generic index split)
  auto load_rows = [&](bf16* dst, int pitch, int rows, int n_first, int col0, int ncol8) {
    if (128 % ncol8 == 0) {
      const int rstep = 128 / ncol8, c = (tid % ncol8) * 8;
      for (int r = tid / ncol8; r < rows; r += rstep) {
        const int n = n_first + r;
        if (n < N) cp_async16(smem_u32(dst + r * pitch + c), qkv + prow(n) * 3 * C + col0 + c);
        else *reinterpret_cast<uint4*>(dst + r * pitch + c) = make_uint4(0u, 0u, 0u, 0u);
      }
    } else {
      for (int i = tid; i < rows * ncol8; i += 128) {
        const int r = i / ncol8, c = (i - r * ncol8) * 8, n = n_first + r;
        if (n < N) cp_async16(smem_u32(dst + r * pitch + c), qkv + prow(n) * 3 * C + col0 + c);
        else *reinterpret_cast<uint4*>(dst + r * pitch + c) = make_uint4(0u, 0u, 0u, 0u);
      }
    }
  };
  load_rows(Qs, qp, S1A_Q, q0, 0, c8);
#pragma unroll
  for (int d = 0; d < S1A_NKB - 1; ++d) {                       // Q rides in the first group
    if (d * S1A_KC < N) load_rows(KV + d * kbuf, qp, S1A_KC, d * S1A_KC, C, c8);
    cp_async_commit();
  }
  float S[S1A_NMAX / 8][4];
#pragma unroll
  for (int i = 0; i < S1A_NMAX / 8; ++i) S[i][0] = S[i][1] = S[i][2] = S[i][3] = 0.f;
  const uint32_t qs_u32 = smem_u32(Qs), kv_u32 = smem_u32(KV), ps_u32 = smem_u32(Ps);
  // ldmatrix lane addressing: A (x4): row (l & 7) + ((l >> 3) & 1) * 8, col (l >> 4) * 8;  B (x2): row l & 7, col ((l >> 3) & 1) * 8
  const int a_row = (lane & 7) + ((lane >> 3) & 1) * 8, a_col = (lane >> 4) * 8;
  const int b_row = lane & 7, b_col = ((lane >> 3) & 1) * 8;
  // ---- phase 1: scores ----
#pragma unroll
  for (int kc = 0; kc < S1A_NMAX / S1A_KC; ++kc) {
    if (kc * S1A_KC < N) {                                      // CTA-uniform
      if ((kc + S1A_NKB - 1) * S1A_KC < N)
        load_rows(KV + ((kc + S1A_NKB - 1) % S1A_NKB) * kbuf, qp, S1A_KC, (kc + S1A_NKB - 1) * S1A_KC, C, c8);
      cp_async_commit();                                        // (possibly empty) group: uniform accounting
      cp_async_wait<S1A_NKB - 1>();
      __syncthreads();
      const uint32_t kb_u32 = kv_u32 + static_cast<uint32_t>((kc % S1A_NKB) * kbuf * 2);
      for (int ks = 0; ks < C / 16; ++ks) {
        uint32_t a0, a1, a2, a3;
        ldsm_x4(qs_u32 + static_cast<uint32_t>(((warp * 16 + a_row) * qp + ks * 16 + a_col) * 2), a0, a1, a2, a3);
#pragma unroll
        for (int nb = 0; nb < S1A_KC / 8; ++nb) {
          uint32_t b0, b1;
          ldmatrix_x2(kb_u32 + static_cast<uint32_t>(((nb * 8 + b_row) * qp + ks * 16 + b_col) * 2), b0, b1);
          mma_bf16_16816(S[kc * (S1A_KC / 8) + nb], a0, a1, a2, a3, b0, b1);
        }
      }
      __syncthreads();                                          // chunk consumed: its buffer may be refilled
    }
  }
  // first V tiles in flight behind the softmax
  const int nvc = (N + S1A_VC - 1) / S1A_VC, ntile = (C / S1A_CB) * nvc;
  auto load_v = [&](int ti) {
    const int cb1 = ti / nvc, vc1 = ti - cb1 * nvc;
    load_rows(KV + (ti % S1A_NVB) * vbuf, vp, S1A_VC, vc1 * S1A_VC, 2 * C + cb1 * S1A_CB, S1A_CB / 8);
  };
#pragma unroll
  for (int d = 0; d < S1A_NVB - 1; ++d) {
    if (d < ntile) load_v(d);
    cp_async_commit();
  }
  // ---- softmax over the keys (w_ = softmax(q k^T C^-1/2), layers.py:175-177); rows g and g + 8 of the warp's 16 ----
  const float scale = rsqrtf(static_cast<float>(C));
  float m0 = -INFINITY, m1 = -INFINITY;
#pragma unroll
  for (int i = 0; i < S1A_NMAX / 8; ++i) {
    const int col = i * 8 + 2 * t;
    S[i][0] = col < N ? S[i][0] * scale : -INFINITY;
    S[i][1] = col + 1 < N ? S[i][1] * scale : -INFINITY;
    S[i][2] = col < N ? S[i][2] * scale : -INFINITY;
    S[i][3] = col + 1 < N ? S[i][3] * scale : -INFINITY;
    m0 = fmaxf(m0, fmaxf(S[i][0], S[i][1]));
    m1 = fmaxf(m1, fmaxf(S[i][2], S[i][3]));
  }
  m0 = fmaxf(m0, __shfl_xor_sync(0xffffffffu, m0, 1)); m0 = fmaxf(m0, __shfl_xor_sync(0xffffffffu, m0, 2));
  m1 = fmaxf(m1, __shfl_xor_sync(0xffffffffu, m1, 1)); m1 = fmaxf(m1, __shfl_xor_sync(0xffffffffu, m1, 2));
  float l0 = 0.f, l1 = 0.f;
#pragma unroll
  for (int i = 0; i < S1A_NMAX / 8; ++i) {
    S[i][0] = expf(S[i][0] - m0); S[i][1] = expf(S[i][1] - m0);
    S[i][2] = expf(S[i][2] - m1); S[i][3] = expf(S[i][3] - m1);
    l0 += S[i][0] + S[i][1];
    l1 += S[i][2] + S[i][3];
  }
  l0 += __shfl_xor_sync(0xffffffffu, l0, 1); l0 += __shfl_xor_sync(0xffffffffu, l0, 2);
  l1 += __shfl_xor_sync(0xffffffffu, l1, 1); l1 += __shfl_xor_sync(0xffffffffu, l1, 2);
  const float i0 = 1.0f / l0, i1 = 1.0f / l1;
#pragma unroll
  for (int i = 0; i < S1A_NMAX / 8; ++i) {
    const int col = i * 8 + 2 * t;
    *reinterpret_cast<__nv_bfloat162*>(Ps + (warp * 16 + g) * pp + col) = __floats2bfloat162_rn(S[i][0] * i0, S[i][1] * i0);
    *reinterpret_cast<__nv_bfloat162*>(Ps + (warp * 16 + g + 8) * pp + col) = __floats2bfloat162_rn(S[i][2] * i1, S[i][3] * i1);
  }
  // ---- phase 2: O = P V, one 128-channel block at a time, V tiles of 64 keys double-buffered ----
  float O[S1A_CB / 8][4];
  for (int ti = 0; ti < ntile; ++ti) {
    const int cb = ti / nvc, vc = ti - cb * nvc;
    if (ti + S1A_NVB - 1 < ntile) load_v(ti + S1A_NVB - 1);
    cp_async_commit();
    cp_async_wait<S1A_NVB - 1>();
    __syncthreads();                                            // tile ti landed (and, first time, P written)
    if (vc == 0) {
#pragma unroll
      for (int i = 0; i < S1A_CB / 8; ++i) O[i][0] = O[i][1] = O[i][2] = O[i][3] = 0.f;
    }
    const uint32_t vb_u32 = kv_u32 + static_cast<uint32_t>((ti % S1A_NVB) * vbuf * 2);
#pragma unroll
    for (int ks = 0; ks < S1A_VC / 16; ++ks) {
      uint32_t a0, a1, a2, a3;
      ldsm_x4(ps_u32 + static_cast<uint32_t>(((warp * 16 + a_row) * pp + vc * S1A_VC + ks * 16 + a_col) * 2), a0, a1, a2, a3);
#pragma unroll
      for (int nb = 0; nb < S1A_CB / 8; ++nb) {
        uint32_t b0, b1;
        // V tile is [key][channel]: the transposing load turns 8 keys x 8 channels into the [n][k] fragment
        ldmatrix_x2_trans(vb_u32 + static_cast<uint32_t>(((ks * 16 + (lane & 7) + ((lane >> 3) & 1) * 8) * vp + nb * 8) * 2), b0, b1);
        mma_bf16_16816(O[nb], a0, a1, a2, a3, b0, b1);
      }
    }
    if (vc == nvc - 1) {
      const int n0 = q0 + warp * 16 + g, n1 = n0 + 8;
#pragma unroll
      for (int nb = 0; nb < S1A_CB / 8; ++nb) {
        const int col = cb * S1A_CB + nb * 8 + 2 * t;
        if (n0 < N) *reinterpret_cast<__nv_bfloat162*>(out + prow(n0) * C + col) = __floats2bfloat162_rn(O[nb][0], O[nb][1]);
        if (n1 < N) *reinterpret_cast<__nv_bfloat162*>(out + prow(n1) * C + col) = __floats2bfloat162_rn(O[nb][2], O[nb][3]);
      }
    }
    __syncthreads();                                            // tile consumed
  }
#endif
}

// conv weight [Cout, Cin, k, k] (fp32 / bf16 / fp16 source already converted to fp32) -> T [CoutPad, k*k*Cin] tap-major
// (bf16, or fp32 rounded to TF32)
template <typename T>
__global__ void s1_pack_weight_kernel(const float* __restrict__ w, T* __restrict__ out, int Cout, int Cin, int taps) {
  const size_t n = static_cast<size_t>(Cout) * Cin * taps;
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < n; i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const int t = static_cast<int>(i % taps);
    const int ci = static_cast<int>((i / taps) % Cin);
    const int co = static_cast<int>(i / (static_cast<size_t>(taps) * Cin));
    out[(static_cast<size_t>(co) * taps + t) * Cin + ci] = s1_round<T>(w[i]);
  }
}

}  // namespace hq
