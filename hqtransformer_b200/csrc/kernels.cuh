// Non-GEMM kernels of the HQ sampling loop: input embedding, LayerNorm, KV-cache attention,
// fused temperature / top-k / top-p / Philox categorical draw.
#pragma once

#include "common.cuh"
#include "../../include/hqgraft.h"

namespace hq {

// ------------------------------------------------------------------------------------------------
// K1: spatial-transformer input token (hierarchical_ar.py:493-499, 506-544 with emb_blocks empty):
//   pos == 0 : x[b] = sos row (class embedding / learned sos / caller-provided override)
//   pos  > 0 : x[b] = mean_5( {E_top[c_t] + P_top[pos-1], E_bot[c_b0..3]} + P_emb[0..4] ), codes of pos-1
// One CTA per batch row.
// ------------------------------------------------------------------------------------------------
struct EmbedArgs {
  float* x;                 // [B, D]
  const float* sos_table;   // cls: [n_classes, D]; uncond: [D]
  const float* sos_override;// optional [B, D]
  const int64_t* cond;      // cls: [B]
  const float* E_top; const float* E_bot; const float* P_top; const float* P_emb;
  const int64_t* codes_top; // [B, S]
  const int64_t* codes_bot; // [B, S, 4]
  int D, S, pos, cond_kind;
  // variants (SURVEY.md 8f-3)
  int emb_kind;             // 0: 'transformer1' (mean of the 5 stack tokens + pos_emb_emb); 1: 'reduce' (hierarchical_ar.py:522-526)
  const float* P_top_h;     // position_embedding == '2d' (:508-514): P_top_h[p / Hpos] + P_top_w[p % Hpos]; else nullptr
  const float* P_top_w;
  int Hpos;
};

__global__ void __launch_bounds__(1024) embed_kernel(int trace_id, EmbedArgs a) {
  TraceScope trace_scope(trace_id);
  pdl_launch_dependents();   // programmatic dependent launch: let the next kernel get resident ...
  pdl_wait();                // ... and wait for the previous kernel's results (no-ops without the launch attribute)
  const int b = blockIdx.x;
  float4* xo = reinterpret_cast<float4*>(a.x + static_cast<size_t>(b) * a.D);
  const int n4 = a.D / 4;
  if (a.pos == 0) {
    const float* src;
    if (a.sos_override != nullptr) src = a.sos_override + static_cast<size_t>(b) * a.D;
    else if (a.cond_kind == HQ_COND_CLS) src = a.sos_table + static_cast<size_t>(a.cond[b]) * a.D;
    else src = a.sos_table;
    const float4* s4 = reinterpret_cast<const float4*>(src);
    for (int i = threadIdx.x; i < n4; i += blockDim.x) xo[i] = s4[i];
    return;
  }
  const int p = a.pos - 1;
  const int64_t ct = a.codes_top[static_cast<size_t>(b) * a.S + p];
  const int64_t* cbp = a.codes_bot + (static_cast<size_t>(b) * a.S + p) * 4;
  const float4* et = reinterpret_cast<const float4*>(a.E_top + static_cast<size_t>(ct) * a.D);
  const bool pos2d = a.P_top_h != nullptr;
  // '2d': the reference splits the position with the number of ROWS OF THE TABLE (sqrt(ctx_len_img)), not the grid width
  const float4* pt = reinterpret_cast<const float4*>(pos2d ? a.P_top_h + static_cast<size_t>(p / a.Hpos) * a.D
                                                           : a.P_top + static_cast<size_t>(p) * a.D);
  const float4* pw = pos2d ? reinterpret_cast<const float4*>(a.P_top_w + static_cast<size_t>(p % a.Hpos) * a.D) : nullptr;
  if (a.emb_kind == 1) {
    // 'reduce': x[d] = E_top[c_t][d] + pos[d] + E_bot[c_b[d % 4]][d / 4]   (rearrange 'B (U L) K -> B U (K L)': K outer)
    const int Dq = a.D / 4;
    const float* ebq[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) ebq[j] = a.E_bot + static_cast<size_t>(cbp[j]) * Dq;
    for (int i = threadIdx.x; i < n4; i += blockDim.x) {
      const float4 t = et[i];
      float4 q = pt[i];
      if (pos2d) { const float4 w = pw[i]; q.x += w.x; q.y += w.y; q.z += w.z; q.w += w.w; }
      // elements 4i .. 4i+3 -> bottom code 0..3, element i of its narrow embedding
      xo[i] = make_float4((t.x + q.x) + ebq[0][i], (t.y + q.y) + ebq[1][i], (t.z + q.z) + ebq[2][i], (t.w + q.w) + ebq[3][i]);
    }
    return;
  }
  const float4* eb[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) eb[j] = reinterpret_cast<const float4*>(a.E_bot + static_cast<size_t>(cbp[j]) * a.D);
  const float4* pe = reinterpret_cast<const float4*>(a.P_emb);
  for (int i = threadIdx.x; i < n4; i += blockDim.x) {
    float4 t = et[i], q = pt[i], e0 = pe[i];
    if (pos2d) { const float4 w = pw[i]; q.x += w.x; q.y += w.y; q.z += w.z; q.w += w.w; }
    float4 acc;
    acc.x = (t.x + q.x) + e0.x; acc.y = (t.y + q.y) + e0.y; acc.z = (t.z + q.z) + e0.z; acc.w = (t.w + q.w) + e0.w;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      float4 e = eb[j][i], pj = pe[(j + 1) * n4 + i];
      acc.x += e.x + pj.x; acc.y += e.y + pj.y; acc.z += e.z + pj.z; acc.w += e.w + pj.w;
    }
    acc.x /= 5.0f; acc.y /= 5.0f; acc.z /= 5.0f; acc.w /= 5.0f;
    xo[i] = acc;
  }
}

// text prefix embedding (sampling.py:187-190): x[b*T + t] = E_txt[ids[b, t]] + P_txt[t]
__global__ void __launch_bounds__(1024)
embed_txt_kernel(int trace_id, float* x, const float* sos_override, const int64_t* ids, const float* E_txt, const float* P_txt,
                 int T, int D) {
  TraceScope trace_scope(trace_id);
  pdl_launch_dependents();   // programmatic dependent launch: let the next kernel get resident ...
  pdl_wait();                // ... and wait for the previous kernel's results (no-ops without the launch attribute)
  const int row = blockIdx.x;  // b*T + t
  const int t = row % T;
  float4* xo = reinterpret_cast<float4*>(x + static_cast<size_t>(row) * D);
  const int n4 = D / 4;
  if (sos_override != nullptr) {
    const float4* s4 = reinterpret_cast<const float4*>(sos_override + static_cast<size_t>(row) * D);
    for (int i = threadIdx.x; i < n4; i += blockDim.x) xo[i] = s4[i];
    return;
  }
  const float4* e = reinterpret_cast<const float4*>(E_txt + static_cast<size_t>(ids[row]) * D);
  const float4* p = reinterpret_cast<const float4*>(P_txt + static_cast<size_t>(t) * D);
  for (int i = threadIdx.x; i < n4; i += blockDim.x) {
    float4 a = e[i], c = p[i];
    xo[i] = make_float4(a.x + c.x, a.y + c.y, a.z + c.z, a.w + c.w);
  }
}

// K11: depth pass-1 inputs (hierarchical_ar.py:701-703): y[b*4 + j] = E_top_depth[c_top[b]] + P_depth[j]
__global__ void __launch_bounds__(1024)
embed_depth_kernel(int trace_id, float* y, const float* E_top_depth, const float* P_depth, const int64_t* codes_top, int S, int pos,
                   int D) {
  TraceScope trace_scope(trace_id);
  pdl_launch_dependents();   // programmatic dependent launch: let the next kernel get resident ...
  pdl_wait();                // ... and wait for the previous kernel's results (no-ops without the launch attribute)
  const int b = blockIdx.x;
  const int64_t ct = codes_top[static_cast<size_t>(b) * S + pos];
  const float4* e = reinterpret_cast<const float4*>(E_top_depth + static_cast<size_t>(ct) * D);
  const float4* p = reinterpret_cast<const float4*>(P_depth);
  const int n4 = D / 4;
  for (int i = threadIdx.x; i < n4; i += blockDim.x) {
    const float4 a = e[i];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float4 c = p[j * n4 + i];
      reinterpret_cast<float4*>(y + (static_cast<size_t>(b) * 4 + j) * D)[i] =
          make_float4(a.x + c.x, a.y + c.y, a.z + c.z, a.w + c.w);
    }
  }
}

// 3-level HQTransformer (SURVEY.md 8f-2), spatial input token (hqtransformer.py:453-487, emb_blocks empty):
//   pos == 0 : x[b] = sos row;  pos > 0 : x[b] = mean_21( {E0[c_top] + P_top[pos-1], E1[c_mid 0..3], E2[c_bot 0..15]} + P_emb[0..20] )
struct Embed3Args {
  float* x;
  const float* sos_table; const float* sos_override; const int64_t* cond;
  const float* E0; const float* E1; const float* E2; const float* P_top; const float* P_emb;
  const int64_t* codes_top;   // [B, S]
  const int64_t* codes_mid;   // [B, S, 4]
  const int64_t* codes_bot;   // [B, S, 16]
  int D, S, pos, cond_kind;
};
__global__ void __launch_bounds__(1024) embed3_kernel(int trace_id, Embed3Args a) {
  TraceScope trace_scope(trace_id);
  pdl_launch_dependents();
  pdl_wait();
  const int b = blockIdx.x;
  float4* xo = reinterpret_cast<float4*>(a.x + static_cast<size_t>(b) * a.D);
  const int n4 = a.D / 4;
  if (a.pos == 0) {
    const float* src;
    if (a.sos_override != nullptr) src = a.sos_override + static_cast<size_t>(b) * a.D;
    else if (a.cond_kind == HQ_COND_CLS) src = a.sos_table + static_cast<size_t>(a.cond[b]) * a.D;
    else src = a.sos_table;
    const float4* s4 = reinterpret_cast<const float4*>(src);
    for (int i = threadIdx.x; i < n4; i += blockDim.x) xo[i] = s4[i];
    return;
  }
  const int p = a.pos - 1;
  __shared__ const float* rows[21];
  if (threadIdx.x < 21) {
    const size_t bp = static_cast<size_t>(b) * a.S + p;
    const int j = threadIdx.x;
    rows[j] = j == 0 ? a.E0 + static_cast<size_t>(a.codes_top[bp]) * a.D
            : j < 5 ? a.E1 + static_cast<size_t>(a.codes_mid[bp * 4 + (j - 1)]) * a.D
                    : a.E2 + static_cast<size_t>(a.codes_bot[bp * 16 + (j - 5)]) * a.D;
  }
  __syncthreads();
  const float4* pt = reinterpret_cast<const float4*>(a.P_top + static_cast<size_t>(p) * a.D);
  const float4* pe = reinterpret_cast<const float4*>(a.P_emb);
  for (int i = threadIdx.x; i < n4; i += blockDim.x) {
    // the order of the reference: cat([e0 + pos, e1.., e2..]) + pos_emb_emb, then mean over the 21 tokens (sequential sum)
    const float4 t = reinterpret_cast<const float4*>(rows[0])[i], q = pt[i], e0 = pe[i];
    float4 acc;
    acc.x = (t.x + q.x) + e0.x; acc.y = (t.y + q.y) + e0.y; acc.z = (t.z + q.z) + e0.z; acc.w = (t.w + q.w) + e0.w;
#pragma unroll 4
    for (int j = 1; j < 21; ++j) {
      const float4 e = reinterpret_cast<const float4*>(rows[j])[i], pj = pe[j * n4 + i];
      acc.x += e.x + pj.x; acc.y += e.y + pj.y; acc.z += e.z + pj.z; acc.w += e.w + pj.w;
    }
    acc.x /= 21.0f; acc.y /= 21.0f; acc.z /= 21.0f; acc.w /= 21.0f;
    xo[i] = acc;
  }
}

// 3-level depth pass 2 input ('parallel-add', hqtransformer.py:521-548): token t of the 4x4 bottom cell (raster order):
//   y[b*16 + t] = E1_depth[c_mid[b, parent(t)]] + P2[t] + E0_depth[c_top[b]],  parent(t) = (row/2)*2 + col/2
__global__ void __launch_bounds__(1024)
embed_depth2_kernel(int trace_id, float* y, const float* E1d, const float* E0d, const float* P2, const int64_t* codes_top,
                    const int64_t* codes_mid, int S, int pos, int D) {
  TraceScope trace_scope(trace_id);
  pdl_launch_dependents();
  pdl_wait();
  const int b = blockIdx.x;
  const size_t bp = static_cast<size_t>(b) * S + pos;
  const float4* e0 = reinterpret_cast<const float4*>(E0d + static_cast<size_t>(codes_top[bp]) * D);
  const float4* em[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) em[j] = reinterpret_cast<const float4*>(E1d + static_cast<size_t>(codes_mid[bp * 4 + j]) * D);
  const float4* p2 = reinterpret_cast<const float4*>(P2);
  const int n4 = D / 4;
  for (int i = threadIdx.x; i < n4; i += blockDim.x) {
    const float4 top = e0[i];
    float4 m[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) m[j] = em[j][i];
#pragma unroll
    for (int t = 0; t < 16; ++t) {
      const float4 mm = m[((t >> 2) >> 1) * 2 + ((t & 3) >> 1)];
      const float4 pp = p2[t * n4 + i];
      // (E1 + P2) + E0: the reference adds the position embedding first, the top-code embedding last (:531-548)
      reinterpret_cast<float4*>(y + (static_cast<size_t>(b) * 16 + t) * D)[i] =
          make_float4((mm.x + pp.x) + top.x, (mm.y + pp.y) + top.y, (mm.z + pp.z) + top.z, (mm.w + pp.w) + top.w);
    }
  }
}

// Shared text prefix (SURVEY.md 8f-4: one prompt sampled N times, e.g. the reference notebook repeats a prompt 8x): the prefill
// ran for image 0 only; its T0 cached key / value rows of every layer and its depth start token are broadcast to images 1..B-1.
// K / V: [L][Bmax][Tc][D]; grid (T0, L, B - 1).
template <typename AT>
__global__ void __launch_bounds__(256)
broadcast_prefix_kernel(int trace_id, AT* K, AT* V, float* yd, int Bmax, int Tc, int D) {
  TraceScope trace_scope(trace_id);
  pdl_launch_dependents();
  pdl_wait();
  const int t = blockIdx.x, l = blockIdx.y, b = blockIdx.z + 1;
  const size_t src = (static_cast<size_t>(l) * Bmax * Tc + t) * D;
  const size_t dst = ((static_cast<size_t>(l) * Bmax + b) * Tc + t) * D;
  constexpr int V8 = 16 / static_cast<int>(sizeof(AT));
  for (int i = threadIdx.x * V8; i < D; i += blockDim.x * V8) {
    *reinterpret_cast<uint4*>(K + dst + i) = *reinterpret_cast<const uint4*>(K + src + i);
    *reinterpret_cast<uint4*>(V + dst + i) = *reinterpret_cast<const uint4*>(V + src + i);
  }
  if (t == 0 && l == 0)
    for (int i = threadIdx.x * 4; i < D; i += blockDim.x * 4)
      *reinterpret_cast<float4*>(yd + static_cast<size_t>(b) * D + i) = *reinterpret_cast<const float4*>(yd + i);
}

// Image completion (hq_run_args.prefix_len = P): the spatial input tokens of the given prefix, all of them in one launch.
//   row r = b * N + t, N = T0 + P - 1 tokens per image:
//   t <  T0 : the conditioning row - `sos` override, E_txt[ids[b, t]] + P_txt[t] (text), sos table (class / unconditional)
//   t >= T0 : the stack of position p = t - T0 (0 .. P - 2), what embed_kernel writes at pos = p + 1
// Every float operation is the one of embed_kernel / embed_txt_kernel, in the same order, so each token is bit-identical
// to the one the step path embeds (the arithmetic is restated here so that those kernels stay exactly as they are).
// One CTA per row.
__global__ void __launch_bounds__(1024)
embed_prefix_kernel(int trace_id, EmbedArgs a, const float* __restrict__ E_txt, const float* __restrict__ P_txt, int T0, int N) {
  TraceScope trace_scope(trace_id);
  pdl_launch_dependents();
  pdl_wait();
  const int row = blockIdx.x;
  const int b = row / N, t = row % N;
  float4* xo = reinterpret_cast<float4*>(a.x + static_cast<size_t>(row) * a.D);
  const int n4 = a.D / 4;
  if (t < T0) {
    const float* src;
    if (a.sos_override != nullptr) {
      src = a.sos_override + (static_cast<size_t>(b) * T0 + t) * a.D;
    } else if (a.cond_kind == HQ_COND_TXT) {
      const float4* e = reinterpret_cast<const float4*>(E_txt + static_cast<size_t>(a.cond[static_cast<size_t>(b) * T0 + t]) * a.D);
      const float4* p = reinterpret_cast<const float4*>(P_txt + static_cast<size_t>(t) * a.D);
      for (int i = threadIdx.x; i < n4; i += blockDim.x) {
        float4 u = e[i], c = p[i];
        xo[i] = make_float4(u.x + c.x, u.y + c.y, u.z + c.z, u.w + c.w);
      }
      return;
    } else if (a.cond_kind == HQ_COND_CLS) {
      src = a.sos_table + static_cast<size_t>(a.cond[b]) * a.D;
    } else {
      src = a.sos_table;
    }
    const float4* s4 = reinterpret_cast<const float4*>(src);
    for (int i = threadIdx.x; i < n4; i += blockDim.x) xo[i] = s4[i];
    return;
  }
  const int p = t - T0;
  const int64_t ct = a.codes_top[static_cast<size_t>(b) * a.S + p];
  const int64_t* cbp = a.codes_bot + (static_cast<size_t>(b) * a.S + p) * 4;
  const float4* et = reinterpret_cast<const float4*>(a.E_top + static_cast<size_t>(ct) * a.D);
  const bool pos2d = a.P_top_h != nullptr;
  const float4* pt = reinterpret_cast<const float4*>(pos2d ? a.P_top_h + static_cast<size_t>(p / a.Hpos) * a.D
                                                           : a.P_top + static_cast<size_t>(p) * a.D);
  const float4* pw = pos2d ? reinterpret_cast<const float4*>(a.P_top_w + static_cast<size_t>(p % a.Hpos) * a.D) : nullptr;
  if (a.emb_kind == 1) {
    const int Dq = a.D / 4;
    const float* ebq[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) ebq[j] = a.E_bot + static_cast<size_t>(cbp[j]) * Dq;
    for (int i = threadIdx.x; i < n4; i += blockDim.x) {
      const float4 u = et[i];
      float4 q = pt[i];
      if (pos2d) { const float4 w = pw[i]; q.x += w.x; q.y += w.y; q.z += w.z; q.w += w.w; }
      xo[i] = make_float4((u.x + q.x) + ebq[0][i], (u.y + q.y) + ebq[1][i], (u.z + q.z) + ebq[2][i], (u.w + q.w) + ebq[3][i]);
    }
    return;
  }
  const float4* eb[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) eb[j] = reinterpret_cast<const float4*>(a.E_bot + static_cast<size_t>(cbp[j]) * a.D);
  const float4* pe = reinterpret_cast<const float4*>(a.P_emb);
  for (int i = threadIdx.x; i < n4; i += blockDim.x) {
    float4 u = et[i], q = pt[i], e0 = pe[i];
    if (pos2d) { const float4 w = pw[i]; q.x += w.x; q.y += w.y; q.z += w.z; q.w += w.w; }
    float4 acc;
    acc.x = (u.x + q.x) + e0.x; acc.y = (u.y + q.y) + e0.y; acc.z = (u.z + q.z) + e0.z; acc.w = (u.w + q.w) + e0.w;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      float4 e = eb[j][i], pj = pe[(j + 1) * n4 + i];
      acc.x += e.x + pj.x; acc.y += e.y + pj.y; acc.z += e.z + pj.z; acc.w += e.w + pj.w;
    }
    acc.x /= 5.0f; acc.y /= 5.0f; acc.z /= 5.0f; acc.w /= 5.0f;
    xo[i] = acc;
  }
}

// The same for the 3-level HQTransformer (T0 = 1): row b * N + t is the sos row (t = 0) or the 21-token stack mean of
// position t - 1, with embed3_kernel's operations and order.
__global__ void __launch_bounds__(1024) embed3_prefix_kernel(int trace_id, Embed3Args a, int N) {
  TraceScope trace_scope(trace_id);
  pdl_launch_dependents();
  pdl_wait();
  const int row = blockIdx.x;
  const int b = row / N, t = row % N;
  float4* xo = reinterpret_cast<float4*>(a.x + static_cast<size_t>(row) * a.D);
  const int n4 = a.D / 4;
  if (t == 0) {
    const float* src;
    if (a.sos_override != nullptr) src = a.sos_override + static_cast<size_t>(b) * a.D;
    else if (a.cond_kind == HQ_COND_CLS) src = a.sos_table + static_cast<size_t>(a.cond[b]) * a.D;
    else src = a.sos_table;
    const float4* s4 = reinterpret_cast<const float4*>(src);
    for (int i = threadIdx.x; i < n4; i += blockDim.x) xo[i] = s4[i];
    return;
  }
  const int p = t - 1;
  __shared__ const float* rows[21];
  if (threadIdx.x < 21) {
    const size_t bp = static_cast<size_t>(b) * a.S + p;
    const int j = threadIdx.x;
    rows[j] = j == 0 ? a.E0 + static_cast<size_t>(a.codes_top[bp]) * a.D
            : j < 5 ? a.E1 + static_cast<size_t>(a.codes_mid[bp * 4 + (j - 1)]) * a.D
                    : a.E2 + static_cast<size_t>(a.codes_bot[bp * 16 + (j - 5)]) * a.D;
  }
  __syncthreads();
  const float4* pt = reinterpret_cast<const float4*>(a.P_top + static_cast<size_t>(p) * a.D);
  const float4* pe = reinterpret_cast<const float4*>(a.P_emb);
  for (int i = threadIdx.x; i < n4; i += blockDim.x) {
    const float4 u = reinterpret_cast<const float4*>(rows[0])[i], q = pt[i], e0 = pe[i];
    float4 acc;
    acc.x = (u.x + q.x) + e0.x; acc.y = (u.y + q.y) + e0.y; acc.z = (u.z + q.z) + e0.z; acc.w = (u.w + q.w) + e0.w;
#pragma unroll 4
    for (int j = 1; j < 21; ++j) {
      const float4 e = reinterpret_cast<const float4*>(rows[j])[i], pj = pe[j * n4 + i];
      acc.x += e.x + pj.x; acc.y += e.y + pj.y; acc.z += e.z + pj.z; acc.w += e.w + pj.w;
    }
    acc.x /= 21.0f; acc.y /= 21.0f; acc.z /= 21.0f; acc.w /= 21.0f;
    xo[i] = acc;
  }
}

// model_type 'top2bot' (hierarchical_ar.py:596-601): input of depth pass c >= 1:
//   y[b] = E[code[b]] + P_depth[c - 1], E = tok_emb_top_depth with the top code (c == 1), tok_emb_bot_depth with bottom
//   code c - 2 otherwise.  `codes` points at the first code (element stride `cstride` int64 between images).
__global__ void __launch_bounds__(1024)
embed_depth_seq_kernel(int trace_id, float* y, const float* E, const float* P_row, const int64_t* codes, int cstride, int D) {
  TraceScope trace_scope(trace_id);
  pdl_launch_dependents();
  pdl_wait();
  const int b = blockIdx.x;
  const int64_t c = codes[static_cast<size_t>(b) * cstride];
  const float4* e = reinterpret_cast<const float4*>(E + static_cast<size_t>(c) * D);
  const float4* p = reinterpret_cast<const float4*>(P_row);
  for (int i = threadIdx.x; i < D / 4; i += blockDim.x) {
    const float4 a = e[i], q = p[i];
    reinterpret_cast<float4*>(y + static_cast<size_t>(b) * D)[i] = make_float4(a.x + q.x, a.y + q.y, a.z + q.z, a.w + q.w);
  }
}

// model_type 'bidirectional' (hierarchical_ar.py:808-811): tokens 1..4 of the five-token depth input are the bare position
// embeddings: y[b*5 + 1 + j] = P_depth[j]  (token 0 = hs + sos_depth is written by the ln_f launch).
__global__ void __launch_bounds__(1024)
depth_pos_rows_kernel(int trace_id, float* y, const float* P_depth, int D) {
  TraceScope trace_scope(trace_id);
  pdl_launch_dependents();
  pdl_wait();
  const int b = blockIdx.x;
  const float4* p = reinterpret_cast<const float4*>(P_depth);
  const int n4 = D / 4;
  for (int i = threadIdx.x; i < n4; i += blockDim.x)
#pragma unroll
    for (int j = 0; j < 4; ++j) reinterpret_cast<float4*>(y + (static_cast<size_t>(b) * 5 + 1 + j) * D)[i] = p[j * n4 + i];
}

// ------------------------------------------------------------------------------------------------
// K2: LayerNorm (eps 1e-5, affine), one warp per row, fp32 statistics (two-pass).
//   out[r * out_mul] = LN(x[(r / in_group) * in_mul + in_off + r % in_group]) * gamma + beta (+ add)    OutT = float | bf16 | f16
// (in_group = out_mul = 1 everywhere except the 'bidirectional' depth pass, whose five-token stacks are normalised by
//  ln_top (token 0) and ln_bot (tokens 1..4) and whose token 0 comes from ln_f of the spatial stream)
// The (+ add) form produces the depth transformer's start token hs + sos_depth (hierarchical_ar.py:561, 685).
// ------------------------------------------------------------------------------------------------
constexpr int LN_THREADS = 128;
constexpr int LN_MAXV = 3;    // float4 per thread held in registers: rows up to 3 * 512 = 1536 columns
constexpr int LN_MAXFOLD = 6; // split-K partial sums a LayerNorm can fold in (kernel instantiated for <= 3 and <= 6)

template <typename OutT>
__device__ __forceinline__ void ln_store4(OutT* o, int i, float y0, float y1, float y2, float y3) {
  if constexpr (sizeof(OutT) == 4) {
    *reinterpret_cast<float4*>(reinterpret_cast<float*>(o) + i) = make_float4(y0, y1, y2, y3);
  } else {
    uint2 u;
    u.x = pack2_rn<OutT>(y0, y1);
    u.y = pack2_rn<OutT>(y2, y3);
    *reinterpret_cast<uint2*>(o + i) = u;
  }
}

__device__ __forceinline__ float block_sum_128(float v, float* red /*[4]*/) {
  v = warp_sum(v);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  return (red[0] + red[1]) + (red[2] + red[3]);
}

// One row per CTA (128 threads).  A decode step is a chain of ~150 dependent kernels, so what matters here is the
// number of serialized memory round trips, not bandwidth: x, gamma, beta (and the optional partial sums / addend)
// are ALL requested before the first use - one round trip - then two block reductions and the stores.
//   fold != nullptr: x[r] += fold_bias + sum_s fold[s][r]  first (split-K partial sums of the preceding GEMM, summed
//   in a fixed order, so the result is deterministic), and the updated x row is written back.
template <typename OutT, int MAXFOLD>
__global__ void __launch_bounds__(LN_THREADS)
layernorm_kernel(int trace_id, float* __restrict__ x, const float* __restrict__ gamma, const float* __restrict__ beta,
                 const float* __restrict__ add, OutT* __restrict__ out, int rows, int D, int in_mul, int in_off,
                 const float* __restrict__ fold, int n_fold, size_t fold_stride, const float* __restrict__ fold_bias,
                 int in_group, int out_mul) {
  TraceScope trace_scope(trace_id);
  pdl_launch_dependents();
  pdl_wait();
  __shared__ float red[4];
  const int r = blockIdx.x;
  const size_t in_row = static_cast<size_t>(r / in_group) * in_mul + in_off + (r % in_group);
  float* xr = x + in_row * D;
  OutT* o = out + static_cast<size_t>(r) * out_mul * D;
  const int tid = threadIdx.x;
  if (D <= LN_MAXV * LN_THREADS * 4) {
    float4 v[LN_MAXV], g[LN_MAXV], bt[LN_MAXV], ad[LN_MAXV], fb[LN_MAXV], f[MAXFOLD][LN_MAXV];
    const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int j = 0; j < LN_MAXV; ++j) {
      const int i = (j * LN_THREADS + tid) * 4;
      const int ic = i < D ? i : 0;                       // clamped: the load is unconditional, the value masked
      v[j] = *reinterpret_cast<const float4*>(xr + ic);
      g[j] = *reinterpret_cast<const float4*>(gamma + ic);
      bt[j] = *reinterpret_cast<const float4*>(beta + ic);
      ad[j] = add != nullptr ? *reinterpret_cast<const float4*>(add + ic) : z4;
      fb[j] = z4;
#pragma unroll
      for (int sidx = 0; sidx < MAXFOLD; ++sidx) f[sidx][j] = z4;
      if (fold != nullptr) {
        const float* fr = fold + in_row * D + ic;
        fb[j] = fold_bias != nullptr ? *reinterpret_cast<const float4*>(fold_bias + ic) : z4;
#pragma unroll
        for (int sidx = 0; sidx < MAXFOLD; ++sidx)
          if (sidx < n_fold) f[sidx][j] = *reinterpret_cast<const float4*>(fr + sidx * fold_stride);
      }
    }
    float s = 0.f;
#pragma unroll
    for (int j = 0; j < LN_MAXV; ++j) {
      const int i = (j * LN_THREADS + tid) * 4;
      if (fold != nullptr) {
        float4 a = f[0][j];                               // fixed left-to-right order: deterministic
#pragma unroll
        for (int sidx = 1; sidx < MAXFOLD; ++sidx) {
          a.x += f[sidx][j].x; a.y += f[sidx][j].y; a.z += f[sidx][j].z; a.w += f[sidx][j].w;
        }
        v[j].x += fb[j].x + a.x;
        v[j].y += fb[j].y + a.y;
        v[j].z += fb[j].z + a.z;
        v[j].w += fb[j].w + a.w;
        if (i < D) *reinterpret_cast<float4*>(xr + i) = v[j];
      }
      if (i < D) s += (v[j].x + v[j].y) + (v[j].z + v[j].w);
    }
    const float mean = block_sum_128(s, red) / static_cast<float>(D);
    float q = 0.f;
#pragma unroll
    for (int j = 0; j < LN_MAXV; ++j) {
      if ((j * LN_THREADS + tid) * 4 < D) {
        const float a = v[j].x - mean, b = v[j].y - mean, c = v[j].z - mean, d = v[j].w - mean;
        q += (a * a + b * b) + (c * c + d * d);
      }
    }
    const float rstd = 1.0f / sqrtf(block_sum_128(q, red) / static_cast<float>(D) + 1e-5f);
#pragma unroll
    for (int j = 0; j < LN_MAXV; ++j) {
      const int i = (j * LN_THREADS + tid) * 4;
      if (i < D) {
        ln_store4<OutT>(o, i, (v[j].x - mean) * rstd * g[j].x + bt[j].x + ad[j].x,
                        (v[j].y - mean) * rstd * g[j].y + bt[j].y + ad[j].y,
                        (v[j].z - mean) * rstd * g[j].z + bt[j].z + ad[j].z,
                        (v[j].w - mean) * rstd * g[j].w + bt[j].w + ad[j].w);
      }
    }
    return;
  }
  // wide rows (D > 1536): strided passes
  if (fold != nullptr) {
    for (int i = tid * 4; i < D; i += LN_THREADS * 4) {
      float4 v = *reinterpret_cast<const float4*>(xr + i);
      const float* fr = fold + in_row * D + i;
      float4 acc = *reinterpret_cast<const float4*>(fr);
      for (int sidx = 1; sidx < n_fold; ++sidx) {
        const float4 f = *reinterpret_cast<const float4*>(fr + sidx * fold_stride);
        acc.x += f.x; acc.y += f.y; acc.z += f.z; acc.w += f.w;
      }
      if (fold_bias != nullptr) {
        const float4 b = *reinterpret_cast<const float4*>(fold_bias + i);
        acc.x += b.x; acc.y += b.y; acc.z += b.z; acc.w += b.w;
      }
      v.x += acc.x; v.y += acc.y; v.z += acc.z; v.w += acc.w;
      *reinterpret_cast<float4*>(xr + i) = v;
    }
    __syncthreads();
  }
  float s = 0.f;
  for (int i = tid * 4; i < D; i += LN_THREADS * 4) {
    const float4 v = *reinterpret_cast<const float4*>(xr + i);
    s += (v.x + v.y) + (v.z + v.w);
  }
  const float mean = block_sum_128(s, red) / static_cast<float>(D);
  float q = 0.f;
  for (int i = tid * 4; i < D; i += LN_THREADS * 4) {
    const float4 v = *reinterpret_cast<const float4*>(xr + i);
    const float a = v.x - mean, b = v.y - mean, c = v.z - mean, d = v.w - mean;
    q += (a * a + b * b) + (c * c + d * d);
  }
  const float rstd = 1.0f / sqrtf(block_sum_128(q, red) / static_cast<float>(D) + 1e-5f);
  for (int i = tid * 4; i < D; i += LN_THREADS * 4) {
    const float4 v = *reinterpret_cast<const float4*>(xr + i);
    const float4 g = *reinterpret_cast<const float4*>(gamma + i);
    const float4 bt = *reinterpret_cast<const float4*>(beta + i);
    float y0 = (v.x - mean) * rstd * g.x + bt.x, y1 = (v.y - mean) * rstd * g.y + bt.y;
    float y2 = (v.z - mean) * rstd * g.z + bt.z, y3 = (v.w - mean) * rstd * g.w + bt.w;
    if (add != nullptr) {
      const float4 a4 = *reinterpret_cast<const float4*>(add + i);
      y0 += a4.x; y1 += a4.y; y2 += a4.z; y3 += a4.w;
    }
    ln_store4<OutT>(o, i, y0, y1, y2, y3);
  }
}

// ------------------------------------------------------------------------------------------------
// K5: attention of new queries over cached keys/values (layers.py:93-187), head size 64.
// One warp per (query row m, head h); 8 lanes x 16 B cover the 128-byte (bf16) head slice of one key, so a
// warp-wide load touches 4 complete keys; fp32 scores / softmax / accumulation.
//   b = m / Tq, i = m % Tq; keys of batch b live at rows b * t_stride + t of K / V (row pitch D)
//   n_keys = causal ? kbase + i + 1 : kbase      (scores scaled by 1/8 = hs^-1/2, layers.py:102)
// Used for: spatial decode (Tq = 1, kbase = t + 1), depth pass 1 (Tq = 4, kbase = 5), text prefill (causal).
// ------------------------------------------------------------------------------------------------
constexpr int ATT_MAX_KEYS = 128;
constexpr int ATT_WARPS = 8;

template <typename AT>
__global__ void __launch_bounds__(ATT_WARPS * 32)
attention_kernel(int trace_id, const AT* __restrict__ q, const AT* __restrict__ K, const AT* __restrict__ V, AT* __restrict__ out,
                 int M, int n_heads, int D, int Tq, int t_stride, int kbase, int causal) {
  TraceScope trace_scope(trace_id);
  pdl_launch_dependents();   // programmatic dependent launch: let the next kernel get resident ...
  pdl_wait();                // ... and wait for the previous kernel's results (no-ops without the launch attribute)
  __shared__ float sc[ATT_WARPS][ATT_MAX_KEYS];
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int item = blockIdx.x * ATT_WARPS + w;
  if (item >= M * n_heads) return;
  const int m = item / n_heads, h = item % n_heads;
  const int b = m / Tq, i = m % Tq;
  const int n_keys = causal ? (kbase + i + 1) : kbase;
  const int g = lane >> 3, c = lane & 7;

  float qv[8];
  load8(q + static_cast<size_t>(m) * D + h * 64 + c * 8, qv);
  const AT* Kb = K + static_cast<size_t>(b) * t_stride * D + h * 64 + c * 8;
  const AT* Vb = V + static_cast<size_t>(b) * t_stride * D + h * 64 + c * 8;

#pragma unroll 4
  for (int tb = 0; tb < n_keys; tb += 4) {     // warp-uniform trip count: the shuffles below need all 32 lanes
    const int t = tb + g;
    float kv[8];
    if (t < n_keys) {
      load8_stream(Kb + static_cast<size_t>(t) * D, kv);
    } else {
#pragma unroll
      for (int e = 0; e < 8; ++e) kv[e] = 0.f;
    }
    float s = 0.f;
#pragma unroll
    for (int e = 0; e < 8; ++e) s = fmaf(qv[e], kv[e] * 0.125f, s);
    s += __shfl_xor_sync(0xffffffffu, s, 1);
    s += __shfl_xor_sync(0xffffffffu, s, 2);
    s += __shfl_xor_sync(0xffffffffu, s, 4);
    if (c == 0 && t < n_keys) sc[w][t] = s;
  }
  __syncwarp();
  float mx = -INFINITY;
  for (int t = lane; t < n_keys; t += 32) mx = fmaxf(mx, sc[w][t]);
  mx = warp_max(mx);
  float sum = 0.f;
  for (int t = lane; t < n_keys; t += 32) {
    const float e = expf(sc[w][t] - mx);
    sc[w][t] = e;
    sum += e;
  }
  sum = warp_sum(sum);
  __syncwarp();
  const float inv = 1.0f / sum;
  float acc[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) acc[e] = 0.f;
#pragma unroll 4
  for (int t = g; t < n_keys; t += 4) {
    float vv[8];
    load8_stream(Vb + static_cast<size_t>(t) * D, vv);
    const float p = sc[w][t] * inv;
#pragma unroll
    for (int e = 0; e < 8; ++e) acc[e] = fmaf(p, vv[e], acc[e]);
  }
#pragma unroll
  for (int e = 0; e < 8; ++e) {
    acc[e] += __shfl_xor_sync(0xffffffffu, acc[e], 8);
    acc[e] += __shfl_xor_sync(0xffffffffu, acc[e], 16);
  }
  if (g == 0) store8(out + static_cast<size_t>(m) * D + h * 64 + c * 8, acc);
}

// ------------------------------------------------------------------------------------------------
// K5b: depth-transformer attention (hierarchical_ar.py:696-710 via layers.py:93-187): a handful of keys (<= 8; the
// parallel depth pass has 4 queries over 5 keys, no mask).  One warp per (query row, head); lane = (key slot g, 16-byte
// piece c).  q, both key rows and both value rows of a lane are requested before anything is used: one memory round
// trip, then shuffles.
// ------------------------------------------------------------------------------------------------
template <typename AT>
__global__ void __launch_bounds__(ATT_WARPS * 32)
attention_fewkeys_kernel(int trace_id, const AT* __restrict__ q, const AT* __restrict__ K, const AT* __restrict__ V,
                         AT* __restrict__ out, int M, int n_heads, int D, int Tq, int t_stride, int n_keys) {
  TraceScope trace_scope(trace_id);
  pdl_launch_dependents();
  pdl_wait();
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int item = blockIdx.x * ATT_WARPS + w;
  if (item >= M * n_heads) return;
  const int m = item / n_heads, h = item % n_heads;
  const int b = m / Tq;
  const int g = lane >> 3, c = lane & 7;
  const size_t base = static_cast<size_t>(b) * t_stride * D + h * 64 + c * 8;
  const int t0 = g, t1 = g + 4;
  const int t0c = t0 < n_keys ? t0 : 0, t1c = t1 < n_keys ? t1 : 0;   // clamped: loads are unconditional
  float qv[8], k0[8], k1[8], v0[8], v1[8];
  load8(q + static_cast<size_t>(m) * D + h * 64 + c * 8, qv);
  load8(K + base + static_cast<size_t>(t0c) * D, k0);
  load8(K + base + static_cast<size_t>(t1c) * D, k1);
  load8(V + base + static_cast<size_t>(t0c) * D, v0);
  load8(V + base + static_cast<size_t>(t1c) * D, v1);
  float s0 = 0.f, s1 = 0.f;
#pragma unroll
  for (int e = 0; e < 8; ++e) {
    s0 = fmaf(qv[e], k0[e] * 0.125f, s0);
    s1 = fmaf(qv[e], k1[e] * 0.125f, s1);
  }
#pragma unroll
  for (int o = 1; o < 8; o <<= 1) {
    s0 += __shfl_xor_sync(0xffffffffu, s0, o);
    s1 += __shfl_xor_sync(0xffffffffu, s1, o);
  }
  if (t0 >= n_keys) s0 = -INFINITY;
  if (t1 >= n_keys) s1 = -INFINITY;
  float mx = fmaxf(s0, s1);
  mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 8));
  mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 16));
  const float e0 = (t0 < n_keys) ? expf(s0 - mx) : 0.f;
  const float e1 = (t1 < n_keys) ? expf(s1 - mx) : 0.f;
  float sum = e0 + e1;                       // identical on the 8 lanes of a key slot
  sum += __shfl_xor_sync(0xffffffffu, sum, 8);
  sum += __shfl_xor_sync(0xffffffffu, sum, 16);
  const float inv = 1.0f / sum;
  const float p0 = e0 * inv, p1 = e1 * inv;
  float acc[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) {
    acc[e] = fmaf(p0, v0[e], p1 * v1[e]);
    acc[e] += __shfl_xor_sync(0xffffffffu, acc[e], 8);
    acc[e] += __shfl_xor_sync(0xffffffffu, acc[e], 16);
  }
  if (g == 0) store8(out + static_cast<size_t>(m) * D + h * 64 + c * 8, acc);
}

// ------------------------------------------------------------------------------------------------
// K5c: the parallel depth pass proper - FOUR queries of one image over its <= 5 depth keys (5 in the reference:
// the pass-0 token and the four pass-1 tokens, no mask; hierarchical_ar.py:696-710).  One warp per (image, head):
// lane = (query g, 16-byte piece c).  Keys and values are fetched once for all four queries (the four lane groups
// read the same addresses: one L1 transaction each), every load of a lane - its q piece, n_keys key pieces, n_keys value
// pieces - is issued before anything is used (one memory round trip), and each lane owns one 16-byte piece of one
// output row, so the value pass needs no cross-lane reduction.
// ------------------------------------------------------------------------------------------------
// 8 consecutive activations kept as loaded (bf16 / fp16: one 16-byte register quad) until they are used
template <typename AT> struct Raw8;
template <> struct Raw8<bf16> {
  uint4 u;
  __device__ __forceinline__ void load(const bf16* p) { u = *reinterpret_cast<const uint4*>(p); }
  __device__ __forceinline__ void get(float (&o)[8]) const {
    const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&u);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float2 f = __bfloat1622float2(h[i]);
      o[2 * i] = f.x;
      o[2 * i + 1] = f.y;
    }
  }
};
template <> struct Raw8<f16> {
  uint4 u;
  __device__ __forceinline__ void load(const f16* p) { u = *reinterpret_cast<const uint4*>(p); }
  __device__ __forceinline__ void get(float (&o)[8]) const {
    const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float2 f = unpack2<f16>(w[i]);
      o[2 * i] = f.x;
      o[2 * i + 1] = f.y;
    }
  }
};
template <> struct Raw8<float> {
  float4 a, b;
  __device__ __forceinline__ void load(const float* p) {
    a = *reinterpret_cast<const float4*>(p);
    b = *reinterpret_cast<const float4*>(p + 4);
  }
  __device__ __forceinline__ void get(float (&o)[8]) const {
    o[0] = a.x; o[1] = a.y; o[2] = a.z; o[3] = a.w; o[4] = b.x; o[5] = b.y; o[6] = b.z; o[7] = b.w;
  }
};

constexpr int ATT_DEPTH_KEYS = 5;   // slots of the depth KV cache: the pass-0 token + the four pass-1 tokens

template <typename AT>
__global__ void __launch_bounds__(ATT_WARPS * 32, 3)
attention_depth4_kernel(int trace_id, const AT* __restrict__ q, const AT* __restrict__ K, const AT* __restrict__ V,
                        AT* __restrict__ out, int B, int n_heads, int D, int t_stride, int n_keys) {
  TraceScope trace_scope(trace_id);
  pdl_launch_dependents();
  pdl_wait();
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int item = blockIdx.x * ATT_WARPS + w;
  if (item >= B * n_heads) return;
  const int b = item / n_heads, h = item % n_heads;
  const int g = lane >> 3, c = lane & 7;
  const size_t qoff = (static_cast<size_t>(b) * 4 + g) * D + h * 64 + c * 8;
  const size_t kbase = static_cast<size_t>(b) * t_stride * D + h * 64 + c * 8;
  Raw8<AT> qr, kr[ATT_DEPTH_KEYS], vr[ATT_DEPTH_KEYS];
  qr.load(q + qoff);
#pragma unroll
  for (int t = 0; t < ATT_DEPTH_KEYS; ++t) {
    const int tc = t < n_keys ? t : 0;               // clamped: loads are unconditional, surplus keys masked below
    kr[t].load(K + kbase + static_cast<size_t>(tc) * D);
    vr[t].load(V + kbase + static_cast<size_t>(tc) * D);
  }
  float qv[8];
  qr.get(qv);
  float s[ATT_DEPTH_KEYS];
  float mx = -INFINITY;
#pragma unroll
  for (int t = 0; t < ATT_DEPTH_KEYS; ++t) {
    float kv[8];
    kr[t].get(kv);
    float d = 0.f;
#pragma unroll
    for (int e = 0; e < 8; ++e) d = fmaf(qv[e], kv[e] * 0.125f, d);
    d += __shfl_xor_sync(0xffffffffu, d, 1);
    d += __shfl_xor_sync(0xffffffffu, d, 2);
    d += __shfl_xor_sync(0xffffffffu, d, 4);
    s[t] = t < n_keys ? d : -INFINITY;
    mx = fmaxf(mx, s[t]);
  }
  float sum = 0.f;
#pragma unroll
  for (int t = 0; t < ATT_DEPTH_KEYS; ++t) {
    s[t] = t < n_keys ? expf(s[t] - mx) : 0.f;
    sum += s[t];
  }
  const float inv = 1.0f / sum;
  float acc[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) acc[e] = 0.f;
#pragma unroll
  for (int t = 0; t < ATT_DEPTH_KEYS; ++t) {
    float vv[8];
    vr[t].get(vv);
    const float p = s[t] * inv;
#pragma unroll
    for (int e = 0; e < 8; ++e) acc[e] = fmaf(p, vv[e], acc[e]);
  }
  store8(out + qoff, acc);
}

// ------------------------------------------------------------------------------------------------
// K5a: single-query attention over the spatial KV cache - the bandwidth-bound kernel of the loop.
// One CTA per (batch row, head group): grid = B * G CTAs, HPC = n_heads / G heads (= consumer warps) each, so that
// the ~1000 small CTAs balance over the 148 SMs (one CTA per image left 40 SMs with half the work of the others).
// A producer warp streams the group's slice of the row's keys and then values - HPC*64 contiguous elements per key -
// through a ring of shared-memory stages with cp.async.bulk (CH keys per stage, completion on mbarriers): no register
// staging, ~4 stages in flight per CTA and 8 CTAs per SM.  All cached keys except the newest one were written by
// earlier launches, so with programmatic dependent launch the producer fills the ring BEFORE griddepcontrol.wait and
// only the chunk holding the newest key (and everything after it) waits for the QKV GEMM.
// Consumer warp = one head; lane = (key slot 0..3, 16-byte piece 0..7).  Scores go to shared memory, a full (not
// online) softmax is taken once all keys are seen - the arithmetic of the reference's bmm / softmax / bmm
// (layers.py:102, 183-186).
// ------------------------------------------------------------------------------------------------
constexpr int ATTD_MAXHPC = 24;   // heads (consumer warps) per CTA
constexpr int ATTD_STAGES = 4;

template <typename AT>
__global__ void __launch_bounds__((ATTD_MAXHPC + 1) * 32)
attention_decode_kernel(int trace_id, const AT* __restrict__ q, const AT* __restrict__ K, const AT* __restrict__ V,
                        AT* __restrict__ out, int D, int t_stride, int n_keys, int CH, int hpc, int groups,
                        int sleep_ns) {
#if defined(__CUDA_ARCH__)
  TraceScope trace_scope(trace_id);
  extern __shared__ __align__(128) uint8_t att_smem[];
  const int slice = hpc * 64;                                       // elements of one key owned by this CTA
  const int row_bytes = slice * static_cast<int>(sizeof(AT));
  const int stage_bytes = CH * row_bytes;
  uint8_t* ring = att_smem;
  float* sc = reinterpret_cast<float*>(att_smem + ATTD_STAGES * stage_bytes);              // [hpc][ATT_MAX_KEYS]
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(sc + hpc * ATT_MAX_KEYS);
  uint64_t* empty_bar = full_bar + ATTD_STAGES;
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int b = blockIdx.x / groups, grp = blockIdx.x % groups;
  const int h0 = grp * hpc;
  const int nck = (n_keys + CH - 1) / CH;

  if (threadIdx.x == 0) {
    phase_mark(0);
    for (int s = 0; s < ATTD_STAGES; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], hpc);
    }
    fence_barrier_init();
  }
  __syncthreads();
  if (threadIdx.x == 0) phase_mark(1);
  pdl_launch_dependents();

  if (w == hpc) {
    // ---- producer: K chunks then V chunks through the ring; one bulk copy per key (slice bytes, contiguous) ----
    if (lane == 0) {
      const AT* Kb = K + static_cast<size_t>(b) * t_stride * D + h0 * 64;
      const AT* Vb = V + static_cast<size_t>(b) * t_stride * D + h0 * 64;
      bool waited = false;
      if (sleep_ns < 0) {        // no prefetch ahead of griddepcontrol.wait
        pdl_wait();
        waited = true;
        sleep_ns = 0;
      }
      for (int i = 0; i < 2 * nck; ++i) {
        const int s = i % ATTD_STAGES;
        const uint32_t ph = (i / ATTD_STAGES) & 1;
        const int ck = i < nck ? i : i - nck;
        const int rows = (n_keys - ck * CH) < CH ? (n_keys - ck * CH) : CH;
        // chunks made of keys older than the newest one do not depend on the previous kernel
        if (!waited && (i >= nck || ck * CH + rows >= n_keys)) {
          pdl_wait();
          waited = true;
        }
        if (sleep_ns) mbar_wait_sleep(&empty_bar[s], ph ^ 1, sleep_ns);
        else mbar_wait(&empty_bar[s], ph ^ 1);
        mbar_arrive_expect_tx(&full_bar[s], static_cast<uint32_t>(rows) * row_bytes);
        const AT* src = (i < nck ? Kb : Vb) + static_cast<size_t>(ck) * CH * D;
        for (int r = 0; r < rows; ++r)
          bulk_load_1d(ring + s * stage_bytes + r * row_bytes, src + static_cast<size_t>(r) * D, row_bytes, &full_bar[s]);
      }
    }
    return;
  }
  if (w > hpc) return;

  // ---- consumers: warp w owns head h0 + w ----
  pdl_wait();
  if (sleep_ns < 0) sleep_ns = 0;
  const int g = lane >> 3, c = lane & 7;
  const int h = h0 + w;
  float qv[8];
  load8(q + static_cast<size_t>(b) * D + h * 64 + c * 8, qv);
#pragma unroll
  for (int e = 0; e < 8; ++e) qv[e] *= 0.125f;     // hs^-1/2 = 2^-3 is exact: same products as scaling K (layers.py:102)
  float* row = sc + w * ATT_MAX_KEYS;
  if (threadIdx.x == 0) phase_mark(2);
  int i = 0;
  for (; i < nck; ++i) {
    const int s = i % ATTD_STAGES;
    if (sleep_ns) mbar_wait_sleep(&full_bar[s], (i / ATTD_STAGES) & 1, sleep_ns);
    else mbar_wait(&full_bar[s], (i / ATTD_STAGES) & 1);
    if (i == 0 && threadIdx.x == 0) phase_mark(3);
    const AT* st = reinterpret_cast<const AT*>(ring + s * stage_bytes) + w * 64 + c * 8;
    for (int kk = 0; kk < CH; kk += 4) {
      const int t = i * CH + kk + g;
      float kv[8];
      if (t < n_keys) {
        load8(st + static_cast<size_t>(kk + g) * slice, kv);
      } else {
#pragma unroll
        for (int e = 0; e < 8; ++e) kv[e] = 0.f;
      }
      float sdot = 0.f;
#pragma unroll
      for (int e = 0; e < 8; ++e) sdot = fmaf(qv[e], kv[e], sdot);
      sdot += __shfl_xor_sync(0xffffffffu, sdot, 1);
      sdot += __shfl_xor_sync(0xffffffffu, sdot, 2);
      sdot += __shfl_xor_sync(0xffffffffu, sdot, 4);
      if (c == 0 && t < n_keys) row[t] = sdot;
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(&empty_bar[s]);
  }
  // ---- softmax over this head's scores ----
  if (threadIdx.x == 0) phase_mark(4);
  float mx = -INFINITY;
  for (int t = lane; t < n_keys; t += 32) mx = fmaxf(mx, row[t]);
  mx = warp_max(mx);
  float sum = 0.f;
  for (int t = lane; t < n_keys; t += 32) {
    const float e = expf(row[t] - mx);
    row[t] = e;
    sum += e;
  }
  const float inv = 1.0f / warp_sum(sum);
  __syncwarp();
  if (threadIdx.x == 0) phase_mark(5);
  float acc[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) acc[e] = 0.f;
  for (; i < 2 * nck; ++i) {
    const int s = i % ATTD_STAGES;
    if (sleep_ns) mbar_wait_sleep(&full_bar[s], (i / ATTD_STAGES) & 1, sleep_ns);
    else mbar_wait(&full_bar[s], (i / ATTD_STAGES) & 1);
    const AT* st = reinterpret_cast<const AT*>(ring + s * stage_bytes) + w * 64 + c * 8;
    const int ck = i - nck;
    for (int kk = 0; kk < CH; kk += 4) {
      const int t = ck * CH + kk + g;
      if (t < n_keys) {
        float vv[8];
        load8(st + static_cast<size_t>(kk + g) * slice, vv);
        const float p = row[t] * inv;
#pragma unroll
        for (int e = 0; e < 8; ++e) acc[e] = fmaf(p, vv[e], acc[e]);
      }
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(&empty_bar[s]);
  }
#pragma unroll
  for (int e = 0; e < 8; ++e) {
    acc[e] += __shfl_xor_sync(0xffffffffu, acc[e], 8);
    acc[e] += __shfl_xor_sync(0xffffffffu, acc[e], 16);
  }
  if (g == 0) store8(out + static_cast<size_t>(b) * D + h * 64 + c * 8, acc);
  if (threadIdx.x == 0) {
    phase_mark(6);
    phase_mark(7);
  }
#endif
}

// ------------------------------------------------------------------------------------------------
// K5a (bf16 / fp16): the same single-query attention as ONE streaming pass, persistent, on the mma.sync register path.
// Measured on the scalar kernel above (profiles/r1_attn_phases.txt): with ~25 MB of bulk copies in flight a request
// takes ~4 us to land, and every point where the computation waits for "all of K" (the softmax between the score pass
// and the value pass, the next item) pays that latency again; its score pass is also issue-bound (3 shuffles per 4 keys).
//   * work item = (image, head group); a CTA takes item blockIdx.x first and then draws further items from a global
//     ticket counter (`sched`), so SMs that finish early take more of them - the ~1000 items of a step balance over the
//     148 SMs whatever CTA -> SM placement the (PDL-overlapped) launch got.  The last CTA to finish re-arms the counter.
//   * a ring stage holds 8 keys AND their 8 values, each fetched by ONE 3-D TMA tile load (box 64 dims x HPC heads x
//     8 cache rows, SWIZZLE_128B) - a per-row bulk copy costs ~45 ns of issue time in the producer thread, which at
//     16 copies per stage was the kernel's start-up and nearly its steady-state limit (profiles/r1_attn_phases.txt).
//     The producer warp streams item after item through the ring without draining; a stage is recycled as soon as
//     its 8 keys are folded in, so the kernel behaves like a pure stream.
//   * consumer warp = one head, ONLINE softmax (running max m, running sum l, rescaled accumulator): per stage
//     scores = mma.m16n8k16(A = 8 keys x 16 dims via ldmatrix.x2, B = q in column 0), then
//     acc = acc * exp(m_old - m_new) + mma.m16n8k8(A = V^T via ldmatrix.x2.trans, B = (p_hi, p_lo) in columns 0 / 1):
//     the bf16 head and tail of the fp32 weight p = exp(s - m_new), so p keeps ~16 mantissa bits (fp16: ~22 near
//     p = 1, an absolute floor below, noted at the split).  out = acc / l.
// Same function as the reference's bmm / softmax / bmm (layers.py:102, 183-186); the online form differs from the
// two-pass form only by fp32 rounding of the rescale factors.  Scores scaled by hs^-1/2 = 2^-3 (exact).
// ------------------------------------------------------------------------------------------------
constexpr int ATTM_CH = 8;         // keys (and values) per ring stage
constexpr int ATTM_MAXSTAGES = 8;

__device__ __forceinline__ void ldmatrix_x2(uint32_t addr, uint32_t& r0, uint32_t& r1) {
#if defined(__CUDA_ARCH__)
  asm volatile("ldmatrix.sync.aligned.m8n8.x2.shared.b16 {%0,%1}, [%2];" : "=r"(r0), "=r"(r1) : "r"(addr));
#endif
}
__device__ __forceinline__ void ldmatrix_x2_trans(uint32_t addr, uint32_t& r0, uint32_t& r1) {
#if defined(__CUDA_ARCH__)
  asm volatile("ldmatrix.sync.aligned.m8n8.x2.trans.shared.b16 {%0,%1}, [%2];" : "=r"(r0), "=r"(r1) : "r"(addr));
#endif
}
// D (16x8 fp32) += A (16x16 bf16, row) * B (16x8 bf16, col)
__device__ __forceinline__ void mma_bf16_16816(float (&c)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0,
                                               uint32_t b1) {
#if defined(__CUDA_ARCH__)
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
#endif
}
// D (16x8 fp32) += A (16x8 bf16, row) * B (8x8 bf16, col)
__device__ __forceinline__ void mma_bf16_1688(float (&c)[4], uint32_t a0, uint32_t a1, uint32_t b0) {
#if defined(__CUDA_ARCH__)
  asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5}, {%6}, {%0,%1,%2,%3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a0), "r"(a1), "r"(b0));
#endif
}

// D (16x8 fp32) += A (16x16 fp16, row) * B (16x8 fp16, col)
__device__ __forceinline__ void mma_f16_16816(float (&c)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0,
                                              uint32_t b1) {
#if defined(__CUDA_ARCH__)
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
#endif
}
// D (16x8 fp32) += A (16x8 fp16, row) * B (8x8 fp16, col)
__device__ __forceinline__ void mma_f16_1688(float (&c)[4], uint32_t a0, uint32_t a1, uint32_t b0) {
#if defined(__CUDA_ARCH__)
  asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5}, {%6}, {%0,%1,%2,%3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a0), "r"(a1), "r"(b0));
#endif
}
// the two forms for the element type AT of the operands
template <typename AT>
__device__ __forceinline__ void mma_16816(float (&c)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0, uint32_t b1) {
  if constexpr (std::is_same<AT, bf16>::value) mma_bf16_16816(c, a0, a1, a2, a3, b0, b1);
  else mma_f16_16816(c, a0, a1, a2, a3, b0, b1);
}
template <typename AT>
__device__ __forceinline__ void mma_1688(float (&c)[4], uint32_t a0, uint32_t a1, uint32_t b0) {
  if constexpr (std::is_same<AT, bf16>::value) mma_bf16_1688(c, a0, a1, b0);
  else mma_f16_1688(c, a0, a1, b0);
}

// AT = bf16 | f16 (the element type of q, K, V and out)
template <typename AT>
__global__ void __launch_bounds__((ATTD_MAXHPC + 1) * 32)
attention_decode_mma_kernel(int trace_id, const __grid_constant__ CUtensorMap tmK, const __grid_constant__ CUtensorMap tmV,
                            int row_base, const AT* __restrict__ q, AT* __restrict__ out, int D, int t_stride, int n_keys,
                            int hpc, int groups, int n_items, int stages, unsigned int* __restrict__ sched) {
#if defined(__CUDA_ARCH__)
  TraceScope trace_scope(trace_id);
  const bool prefetch = stages > 0;      // stages < 0: no tile load ahead of griddepcontrol.wait
  if (stages < 0) stages = -stages;
  extern __shared__ uint8_t att_smem_raw[];
  uint8_t* ring = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(att_smem_raw) + 1023) & ~static_cast<uintptr_t>(1023));
  const int slice_bytes = hpc * 128;                                // one key row of this head group
  const int tile_bytes = ATTM_CH * slice_bytes;                     // 8 keys (or values) x hpc heads x 128 B, 1 KB multiple
  const int stage_bytes = 2 * tile_bytes;                           // K tile, then V tile
  uint8_t* qbuf = ring + stages * stage_bytes;                      // [2][slice_bytes]
  float* ostage = reinterpret_cast<float*>(qbuf + 2 * slice_bytes); // [hpc][64] output staging
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(ostage + hpc * 64);
  uint64_t* empty_bar = full_bar + ATTM_MAXSTAGES;
  uint64_t* qfull_bar = empty_bar + ATTM_MAXSTAGES;                 // [2]
  uint64_t* qempty_bar = qfull_bar + 2;                             // [2]
  int* qitem = reinterpret_cast<int*>(qempty_bar + 2);              // [2] item id that goes with qbuf[i]; -1 = no more
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nck = (n_keys + ATTM_CH - 1) / ATTM_CH;
  if (threadIdx.x == 0) {
    phase_mark(0);
    tma_prefetch_desc(&tmK);
    tma_prefetch_desc(&tmV);
    for (int s = 0; s < stages; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], hpc);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(&qfull_bar[s], 1);
      mbar_init(&qempty_bar[s], hpc);
    }
    fence_barrier_init();
  }
  __syncthreads();
  if (threadIdx.x == 0) phase_mark(1);
  pdl_launch_dependents();

  if (w == hpc) {
    // ---- producer: two tensor-tile loads per stage (8 keys x hpc heads, 8 values x hpc heads) ----
    if (lane == 0) {
      bool waited = false;
      int item = blockIdx.x;
      uint32_t g = 0;                                               // ring stages issued so far (all items)
      for (int it = 0;; ++it) {
        const int ip = it & 1;
        const bool have = item < n_items;
        const int b = have ? item / groups : 0, grp = have ? item % groups : 0;
        const int row0 = row_base + b * t_stride;
        auto issue = [&](int ck, int s) {
          mbar_arrive_expect_tx(&full_bar[s], static_cast<uint32_t>(stage_bytes));   // boxes always land whole
          uint8_t* dst = ring + s * stage_bytes;
          tma_load_3d(dst, &tmK, &full_bar[s], 0, grp * hpc, row0 + ck * ATTM_CH);
          tma_load_3d(dst + tile_bytes, &tmV, &full_bar[s], 0, grp * hpc, row0 + ck * ATTM_CH);
        };
        int i = 0;
        if (have && !waited && prefetch) {
          // every key but the newest was written by earlier launches: those stages do not wait for the QKV GEMM
          for (; i < nck - 1 && i < stages; ++i, ++g) issue(i, g % stages);
        }
        if (!waited) {
          pdl_wait();
          waited = true;
        }
        // q slice + item id of this item (or the end marker)
        mbar_wait(&qempty_bar[ip], ((it >> 1) & 1) ^ 1);
        qitem[ip] = have ? item : -1;
        if (!have) {
          mbar_arrive(&qfull_bar[ip]);
          break;
        }
        if (it == 0) {
          mbar_arrive(&qfull_bar[ip]);      // first item: the consumers fetch q themselves
        } else {
          mbar_arrive_expect_tx(&qfull_bar[ip], slice_bytes);
          bulk_load_1d(qbuf + ip * slice_bytes, q + static_cast<size_t>(b) * D + grp * hpc * 64, slice_bytes, &qfull_bar[ip]);
        }
        const int next = static_cast<int>(atomicAdd(sched, 1u)) + static_cast<int>(gridDim.x);
        for (; i < nck; ++i, ++g) {
          const int s = g % stages;
          mbar_wait(&empty_bar[s], ((g / stages) & 1) ^ 1);
          issue(i, s);
        }
        item = next;
      }
      // the last CTA to run out of work re-arms the ticket counter for the next launch
      if (atomicAdd(sched + 1, 1u) == gridDim.x - 1) {
        sched[0] = 0;
        sched[1] = 0;
        __threadfence();
      }
    }
    return;
  }
  if (w > hpc) return;

  // ---- consumers: warp w owns head grp * hpc + w of every item this CTA takes ----
  pdl_wait();
  const int gq = lane >> 2, tq = lane & 3;          // mma fragment coordinates: row / column pair
  const int lr = lane & 7, lm = (lane >> 3) & 1;    // ldmatrix.x2: row within the matrix, matrix index (lanes 0-15)
  const uint32_t ring_u32 = smem_u32(ring);
  // SWIZZLE_128B tile: the 128-byte line of (key lr, head w) is line lr*hpc + w; its 16-byte chunk c sits at
  // c ^ (line & 7).  Step j (16 dims) of this lane's matrix (dims 0-7 | 8-15 -> lm) is chunk 2j + lm.
  // K: matrices feed fragments a0 | a2 (rows 8-15 of the MMA stay zero); V: transposed on load -> a0 | a1.
  uint32_t frag_off[4];
  {
    const uint32_t line = static_cast<uint32_t>(lr * hpc + w);
#pragma unroll
    for (int j = 0; j < 4; ++j) frag_off[j] = line * 128u + (((2u * j + lm) ^ (line & 7u)) << 4);
  }
  float* orow = ostage + w * 64;
  uint32_t g = 0;
  for (int it = 0;; ++it) {
    const int ip = it & 1;
    mbar_wait(&qfull_bar[ip], (it >> 1) & 1);
    const int item = qitem[ip];
    if (item < 0) break;
    // q as the B operand: column 0 (lanes 0-3) holds dims 2*tq, 2*tq+1 (+8) of each 16-dim step
    uint32_t qb[4][2];
    {
      const uint32_t* q32 =
          it == 0 ? reinterpret_cast<const uint32_t*>(q + static_cast<size_t>(item / groups) * D + ((item % groups) * hpc + w) * 64)
                  : reinterpret_cast<const uint32_t*>(qbuf + ip * slice_bytes + w * 128);
#pragma unroll
      for (int ks = 0; ks < 4; ++ks) {
        qb[ks][0] = gq == 0 ? q32[ks * 8 + tq] : 0u;
        qb[ks][1] = gq == 0 ? q32[ks * 8 + 4 + tq] : 0u;
      }
    }
    if (it == 0 && threadIdx.x == 0) phase_mark(2);
    __syncwarp();
    if (lane == 0) mbar_arrive(&qempty_bar[ip]);

    float m_run = -INFINITY, l_run = 0.f;
    float o[4][4];
#pragma unroll
    for (int mt = 0; mt < 4; ++mt)
#pragma unroll
      for (int e = 0; e < 4; ++e) o[mt][e] = 0.f;

    for (int c = 0; c < nck; ++c, ++g) {
      const int s = g % stages;
      const int left = n_keys - c * ATTM_CH;          // valid keys in this stage (>= 1)
      mbar_wait(&full_bar[s], (g / stages) & 1);
      if (g == 0 && threadIdx.x == 0) phase_mark(3);
      const uint32_t kbase = ring_u32 + s * stage_bytes;
      const uint32_t vbase = kbase + tile_bytes;
      // ---- scores of the 8 keys: lane (gq, tq = 0) gets key gq ----
      float sc[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
      for (int ks = 0; ks < 4; ++ks) {
        uint32_t a0, a2;
        ldmatrix_x2(kbase + frag_off[ks], a0, a2);
        mma_16816<AT>(sc, a0, 0u, a2, 0u, qb[ks][0], qb[ks][1]);
      }
      float sk = __shfl_sync(0xffffffffu, sc[0], lane & ~3) * 0.125f;   // every lane of quad gq: score of key gq
      if (gq >= left) sk = -INFINITY;                                    // rows past the cache end are not keys
      float cm = sk;
      cm = fmaxf(cm, __shfl_xor_sync(0xffffffffu, cm, 4));
      cm = fmaxf(cm, __shfl_xor_sync(0xffffffffu, cm, 8));
      cm = fmaxf(cm, __shfl_xor_sync(0xffffffffu, cm, 16));
      const float m_new = fmaxf(m_run, cm);
      const float alpha = expf(m_run - m_new);         // first stage: exp(-inf) = 0
      const float pk = expf(sk - m_new);               // masked keys: exp(-inf) = 0
      float ps = pk;
      ps += __shfl_xor_sync(0xffffffffu, ps, 4);
      ps += __shfl_xor_sync(0xffffffffu, ps, 8);
      ps += __shfl_xor_sync(0xffffffffu, ps, 16);
      l_run = l_run * alpha + ps;
      m_run = m_new;
      // ---- B operand of the value MMA: keys 2*tq, 2*tq+1; column 0 = AT head of p, column 1 = AT tail ----
      // fp16: the tail lies below the normal range (2^-14) for every p < 1/4, so it is rounded on the subnormal grid (spacing
      // 2^-24): head + tail carry p to an absolute ~2^-25 (~3e-8; weights below that vanish), not to a relative 2^-22 -
      // at most ~3e-8 per key next to l_run >= 1.
      const float p0 = __shfl_sync(0xffffffffu, pk, 8 * tq);
      const float p1 = __shfl_sync(0xffffffffu, pk, 8 * tq + 4);
      uint32_t pb = 0u;
      {
        uint32_t h = pack2_rn<AT>(p0, p1);
        if (gq == 1) {
          const float2 f = unpack2<AT>(h);
          h = pack2_rn<AT>(p0 - f.x, p1 - f.y);
        }
        if (gq < 2) pb = h;
      }
      // value rows past the cache end (other cache slots, or whatever the allocation held): 0 * NaN must not
      // reach the accumulator
      uint32_t vmask = 0xFFFFFFFFu;
      if (left < ATTM_CH) vmask = (2 * tq < left ? 0x0000FFFFu : 0u) | (2 * tq + 1 < left ? 0xFFFF0000u : 0u);
      if (alpha != 1.0f) {
#pragma unroll
        for (int mt = 0; mt < 4; ++mt)
#pragma unroll
          for (int e = 0; e < 4; ++e) o[mt][e] *= alpha;
      }
#pragma unroll
      for (int mt = 0; mt < 4; ++mt) {
        uint32_t a0, a1;
        ldmatrix_x2_trans(vbase + frag_off[mt], a0, a1);
        mma_1688<AT>(o[mt], a0 & vmask, a1 & vmask, pb);
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(&empty_bar[s]);
    }
    // ---- out: lanes with tq == 0 hold dims mt*16 + gq (columns 0 + 1) and mt*16 + 8 + gq ----
    const float inv = 1.0f / l_run;
    if (tq == 0) {
#pragma unroll
      for (int mt = 0; mt < 4; ++mt) {
        orow[mt * 16 + gq] = (o[mt][0] + o[mt][1]) * inv;
        orow[mt * 16 + 8 + gq] = (o[mt][2] + o[mt][3]) * inv;
      }
    }
    __syncwarp();
    if (lane < 8) {
      const int b = item / groups, h = (item % groups) * hpc + w;
      float v[8];
      const float4 x0 = *reinterpret_cast<const float4*>(orow + lane * 8);
      const float4 x1 = *reinterpret_cast<const float4*>(orow + lane * 8 + 4);
      v[0] = x0.x; v[1] = x0.y; v[2] = x0.z; v[3] = x0.w; v[4] = x1.x; v[5] = x1.y; v[6] = x1.z; v[7] = x1.w;
      store8(out + static_cast<size_t>(b) * D + h * 64 + lane * 8, v);
    }
    __syncwarp();
    if (it == 0 && threadIdx.x == 0) phase_mark(6);
  }
  if (threadIdx.x == 0) phase_mark(7);
#endif
}

// ------------------------------------------------------------------------------------------------
// Causal attention of the image-completion prefix pass (2-byte engines): the Tq = T0 + P - 1 <= 128 prefix tokens of an
// image, query i over cache slots 0 .. i - attention_kernel with causal = 1, kbase = 0.  attention_kernel gives every
// (query, head) a warp of its own, which re-reads the image's keys and values from L2 once per query; here one CTA per
// (image, head) stages them in shared memory once.  Warp w owns queries 16w .. 16w + 15:
//   S = q K^T on mma.sync m16n8k16 (fp32 accumulation), scaled by 2^-3;
//   fp32 causal softmax in registers (row max / sum over the four lanes of a fragment row);
//   O = P V on mma.sync m16n8k16 with P split into a 2-byte head and tail (attention_decode_mma_kernel's split: P carried
//   to ~2^-17 relative, not the 2-byte type's 2^-8 / 2^-11), then O / sum rounded to the 2-byte type.
// q / out: row b * Tq + i of [*, D]; K / V: row b * t_stride + t of [*, D] (one layer's cache).  Grid: B * n_heads CTAs.
// ------------------------------------------------------------------------------------------------
constexpr int ATTP_PITCH = 72;    // shared row pitch of K / V (elements): 144-byte rows keep fragment loads conflict-free

template <typename AT>
__global__ void __launch_bounds__(256)
attention_prefix_kernel(int trace_id, const AT* __restrict__ q, const AT* __restrict__ K, const AT* __restrict__ V,
                        AT* __restrict__ out, int n_heads, int D, int Tq, int t_stride) {
#if defined(__CUDA_ARCH__)
  TraceScope trace_scope(trace_id);
  pdl_launch_dependents();
  pdl_wait();
  __shared__ __align__(16) AT ks[ATT_MAX_KEYS * ATTP_PITCH];
  __shared__ __align__(16) AT vs[ATT_MAX_KEYS * ATTP_PITCH];
  const int b = blockIdx.x / n_heads, h = blockIdx.x % n_heads;
  // keys staged: Tq rounded up to the 16-key step of the value MMA; rows past Tq are zero (0 * garbage must not reach O)
  const int nrows = (Tq + 15) & ~15;
  const AT* Kb = K + static_cast<size_t>(b) * t_stride * D + h * 64;
  const AT* Vb = V + static_cast<size_t>(b) * t_stride * D + h * 64;
  for (int i = threadIdx.x; i < nrows * 8; i += blockDim.x) {
    const int t = i >> 3, c = (i & 7) * 8;
    uint4 kv = make_uint4(0u, 0u, 0u, 0u), vv = kv;
    if (t < Tq) {
      kv = *reinterpret_cast<const uint4*>(Kb + static_cast<size_t>(t) * D + c);
      vv = *reinterpret_cast<const uint4*>(Vb + static_cast<size_t>(t) * D + c);
    }
    *reinterpret_cast<uint4*>(ks + t * ATTP_PITCH + c) = kv;
    *reinterpret_cast<uint4*>(vs + t * ATTP_PITCH + c) = vv;
  }
  __syncthreads();
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int r0 = w * 16;
  if (r0 >= Tq) return;
  const int gq = lane >> 2, tq = lane & 3;          // fragment row / column pair
  const int ra = r0 + gq, rb = ra + 8;              // the two query rows of this lane
  const int nks = ((r0 + 16 < Tq ? r0 + 16 : Tq) + 15) >> 4;   // 16-key steps holding keys <= the warp's last query

  // q as the A operand (a0 / a2: row ra, a1 / a3: row rb; dims 2tq, 2tq + 1 and + 8 of each 16-dim step)
  uint32_t qa[4][4];
  {
    const uint32_t* qra = reinterpret_cast<const uint32_t*>(q + (static_cast<size_t>(b) * Tq + (ra < Tq ? ra : 0)) * D + h * 64);
    const uint32_t* qrb = reinterpret_cast<const uint32_t*>(q + (static_cast<size_t>(b) * Tq + (rb < Tq ? rb : 0)) * D + h * 64);
#pragma unroll
    for (int kk = 0; kk < 4; ++kk) {
      qa[kk][0] = ra < Tq ? qra[kk * 8 + tq] : 0u;
      qa[kk][1] = rb < Tq ? qrb[kk * 8 + tq] : 0u;
      qa[kk][2] = ra < Tq ? qra[kk * 8 + 4 + tq] : 0u;
      qa[kk][3] = rb < Tq ? qrb[kk * 8 + 4 + tq] : 0u;
    }
  }
  // ---- scores: tile j = keys 8j .. 8j + 7; lane holds (ra | rb, keys 8j + 2tq, 8j + 2tq + 1) ----
  float s[16][4];
#pragma unroll
  for (int j = 0; j < 16; ++j) {
#pragma unroll
    for (int e = 0; e < 4; ++e) s[j][e] = 0.f;
    if (j < 2 * nks) {
      const uint32_t* krow = reinterpret_cast<const uint32_t*>(ks + (j * 8 + gq) * ATTP_PITCH);
#pragma unroll
      for (int kk = 0; kk < 4; ++kk)
        mma_16816<AT>(s[j], qa[kk][0], qa[kk][1], qa[kk][2], qa[kk][3], krow[kk * 8 + tq], krow[kk * 8 + 4 + tq]);
    }
  }
  // ---- causal softmax, fp32 ----
  float mx_a = -INFINITY, mx_b = -INFINITY;
#pragma unroll
  for (int j = 0; j < 16; ++j)
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int key = j * 8 + 2 * tq + (e & 1);
      const int row = e < 2 ? ra : rb;
      const float v = (j < 2 * nks && key <= row) ? s[j][e] * 0.125f : -INFINITY;
      s[j][e] = v;
      if (e < 2) mx_a = fmaxf(mx_a, v);
      else mx_b = fmaxf(mx_b, v);
    }
  mx_a = fmaxf(mx_a, __shfl_xor_sync(0xffffffffu, mx_a, 1));
  mx_a = fmaxf(mx_a, __shfl_xor_sync(0xffffffffu, mx_a, 2));
  mx_b = fmaxf(mx_b, __shfl_xor_sync(0xffffffffu, mx_b, 1));
  mx_b = fmaxf(mx_b, __shfl_xor_sync(0xffffffffu, mx_b, 2));
  float sum_a = 0.f, sum_b = 0.f;
#pragma unroll
  for (int j = 0; j < 16; ++j)
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const float p = expf(s[j][e] - (e < 2 ? mx_a : mx_b));    // masked keys: exp(-inf) = 0
      s[j][e] = p;
      if (e < 2) sum_a += p;
      else sum_b += p;
    }
  sum_a += __shfl_xor_sync(0xffffffffu, sum_a, 1);
  sum_a += __shfl_xor_sync(0xffffffffu, sum_a, 2);
  sum_b += __shfl_xor_sync(0xffffffffu, sum_b, 1);
  sum_b += __shfl_xor_sync(0xffffffffu, sum_b, 2);
  // ---- O = P V: A = P (rows ra | rb, keys 16kk ..), head then tail; B = V rows by ldmatrix.trans ----
  float o[8][4];
#pragma unroll
  for (int nt = 0; nt < 8; ++nt)
#pragma unroll
    for (int e = 0; e < 4; ++e) o[nt][e] = 0.f;
  const uint32_t vrow = smem_u32(vs) + static_cast<uint32_t>((lane & 15) * ATTP_PITCH * 2);
#pragma unroll
  for (int kk = 0; kk < 8; ++kk) {
    if (kk < nks) {
      // a0: (ra, keys 16kk + 2tq ..), a1: (rb, same keys), a2 / a3: keys + 8 - C fragments of tiles 2kk and 2kk + 1
      uint32_t hd[4], tl[4];
#pragma unroll
      for (int r = 0; r < 4; ++r) {
        const int j = 2 * kk + (r >> 1), e = (r & 1) * 2;
        hd[r] = pack2_rn<AT>(s[j][e], s[j][e + 1]);
        const float2 f = unpack2<AT>(hd[r]);
        tl[r] = pack2_rn<AT>(s[j][e] - f.x, s[j][e + 1] - f.y);
      }
#pragma unroll
      for (int nt = 0; nt < 8; ++nt) {
        uint32_t b0, b1;
        ldmatrix_x2_trans(vrow + static_cast<uint32_t>((kk * 16 * ATTP_PITCH + nt * 8) * 2), b0, b1);
        mma_16816<AT>(o[nt], hd[0], hd[1], hd[2], hd[3], b0, b1);
        mma_16816<AT>(o[nt], tl[0], tl[1], tl[2], tl[3], b0, b1);
      }
    }
  }
  const float inv_a = 1.0f / sum_a, inv_b = 1.0f / sum_b;
  AT* oa = out + (static_cast<size_t>(b) * Tq + ra) * D + h * 64 + 2 * tq;
  AT* ob = out + (static_cast<size_t>(b) * Tq + rb) * D + h * 64 + 2 * tq;
#pragma unroll
  for (int nt = 0; nt < 8; ++nt) {
    if (ra < Tq) *reinterpret_cast<uint32_t*>(oa + nt * 8) = pack2_rn<AT>(o[nt][0] * inv_a, o[nt][1] * inv_a);
    if (rb < Tq) *reinterpret_cast<uint32_t*>(ob + nt * 8) = pack2_rn<AT>(o[nt][2] * inv_b, o[nt][3] * inv_b);
  }
#endif
}

// ------------------------------------------------------------------------------------------------
// K10: Sample(z; T, k, p) fused into one kernel per logits row (hierarchical_ar.py:762-785,
// utils/sampling.py:12-37): z /= T; keep z >= k-th largest (ties kept); softmax; nucleus cut on the
// *preceding* cumulative mass; renormalise; one categorical draw.
// No sort: the k-th largest logit and the nucleus boundary are found by bitwise bisection on the
// order-preserving integer image of the floats (32 block-wide count / mass reductions each); the draw is an
// inverse-CDF walk in index order with ONE Philox4x32-10 uniform per row.
// Thread t owns the contiguous slice [t * ipt, (t + 1) * ipt) of the row (registers).
// ------------------------------------------------------------------------------------------------
constexpr int SMP_IPT = 32;

struct SampleArgs {
  const float* logits;  // [R, ldl]
  int ldl, V, R;
  int rows_per_b;       // 1 (top) | 4 (bottom)
  int slot0;            // 0 (top) | 1 (bottom): Philox slot / logits_out slot of the first row of a batch element
  const hq_sampling_params* sp;  // device copy
  int pos, S;
  int64_t* dst_codes;   // code array the draws go to: [B, S, dst_w]
  int dst_w;            // 1 (top codes), 4 (bottom codes of the 2-level model / middle codes), 16 (3-level bottom codes)
  int n_slots;          // stack size (5 | 21): slot stride of logits_out
  int forced;           // 1: codes are given (teacher forcing): leave them untouched
  float* logits_out;    // optional [B, S, 5, Vmax]
  int Vmax;
  int temp_sel;         // which softmax temperature: 0 = top, 1 = bottom, 2 = middle (3-level model)
  int filt_sel;         // which top-k / top-p pair:  0 = top, 1 = bottom, 2 = middle
  int bot_slot;         // rows_per_b == 1 only: >= 0 -> the code goes to dst_codes[b, pos, bot_slot] ('top2bot' passes 1..4)
  float* probs_out;     // optional [R, V] (debug)
  int64_t* flat_out;    // optional [R] (debug)
  // debug overrides (sp == nullptr)
  float temperature, top_p; int top_k; uint64_t seed, row_offset;
};

__device__ __forceinline__ uint32_t float_order_key(float f) {
  const uint32_t b = __float_as_uint(f);
  return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}

template <typename T, typename Op>
__device__ __forceinline__ T block_reduce(T v, Op op, T identity, T* scratch /*[33]*/) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = blockDim.x >> 5;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = op(v, __shfl_xor_sync(0xffffffffu, v, o));
  __syncthreads();  // every thread has consumed scratch[32] of the previous reduction
  if (lane == 0) scratch[w] = v;
  __syncthreads();
  if (w == 0) {
    T r = lane < nw ? scratch[lane] : identity;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) r = op(r, __shfl_xor_sync(0xffffffffu, r, o));
    if (lane == 0) scratch[32] = r;
  }
  __syncthreads();
  return scratch[32];
}

struct OpSumF { __device__ float operator()(float a, float b) const { return a + b; } };
struct OpMaxF { __device__ float operator()(float a, float b) const { return fmaxf(a, b); } };
struct OpSumI { __device__ int operator()(int a, int b) const { return a + b; } };
struct OpMaxI { __device__ int operator()(int a, int b) const { return a > b ? a : b; } };
struct OpMinI { __device__ int operator()(int a, int b) const { return a < b ? a : b; } };

template <int NTHR>
__global__ void __launch_bounds__(NTHR, NTHR == 256 ? 4 : 1) sample_kernel(int trace_id, SampleArgs a) {
  TraceScope trace_scope(trace_id);
  pdl_launch_dependents();   // programmatic dependent launch: let the next kernel get resident ...
  pdl_wait();                // ... and wait for the previous kernel's results (no-ops without the launch attribute)
  __shared__ float fscratch[33];
  __shared__ int iscratch[33];
  __shared__ float wsum[33];
  const int r = blockIdx.x;
  const int b = r / a.rows_per_b, jj = r % a.rows_per_b;
  const int slot = a.slot0 + jj;
  const int tid = threadIdx.x, nthr = blockDim.x;
  const int V = a.V;
  int ipt = (V + nthr - 1) / nthr;
  ipt = (ipt + 3) & ~3;
  const int base = tid * ipt;
  const float* row = a.logits + static_cast<size_t>(r) * a.ldl;

  float temperature, top_p; int top_k; uint64_t seed, row_offset;
  if (a.sp != nullptr) {
    temperature = a.temp_sel == 0 ? a.sp->temperature_top : (a.temp_sel == 1 ? a.sp->temperature_bot : a.sp->temperature_mid);
    top_p = a.filt_sel == 0 ? a.sp->top_p_top : (a.filt_sel == 1 ? a.sp->top_p_bot : a.sp->top_p_mid);
    top_k = a.filt_sel == 0 ? a.sp->top_k_top : (a.filt_sel == 1 ? a.sp->top_k_bot : a.sp->top_k_mid);
    seed = a.sp->seed; row_offset = a.sp->row_offset;
  } else {
    temperature = a.temperature; top_p = a.top_p; top_k = a.top_k; seed = a.seed; row_offset = a.row_offset;
  }

  float z[SMP_IPT];
#pragma unroll
  for (int i = 0; i < SMP_IPT; i += 4) {
    float4 v = make_float4(-INFINITY, -INFINITY, -INFINITY, -INFINITY);
    if (i < ipt && base + i < V) v = *reinterpret_cast<const float4*>(row + base + i);
    z[i] = v.x; z[i + 1] = v.y; z[i + 2] = v.z; z[i + 3] = v.w;
  }
  if (a.logits_out != nullptr) {
    float* lo = a.logits_out + ((static_cast<size_t>(b) * a.S + a.pos) * a.n_slots + slot) * a.Vmax;
#pragma unroll
    for (int i = 0; i < SMP_IPT; ++i)
      if (i < ipt && base + i < V) lo[base + i] = z[i];
  }
  if (a.forced) return;

  if (temperature != 1.0f) {   // z / 1 is the identity: skip 32 fp32 divisions per thread in the default protocol
#pragma unroll
    for (int i = 0; i < SMP_IPT; ++i) z[i] = z[i] / temperature;   // -inf padding stays -inf (T > 0)
  }

  int64_t* dst = a.flat_out != nullptr
                     ? a.flat_out + r
                     : a.dst_codes + (static_cast<size_t>(b) * a.S + a.pos) * a.dst_w +
                           (a.rows_per_b == 1 ? (a.bot_slot < 0 ? 0 : a.bot_slot) : jj);

  // ---- greedy: lowest index among the maxima ----
  float mx = -INFINITY;
#pragma unroll
  for (int i = 0; i < SMP_IPT; ++i) mx = fmaxf(mx, z[i]);
  mx = block_reduce(mx, OpMaxF(), -INFINITY, fscratch);
  if (top_k == 1) {
    int idx = 0x7fffffff;
#pragma unroll
    for (int i = SMP_IPT - 1; i >= 0; --i)
      if (i < ipt && base + i < V && z[i] == mx) idx = base + i;
    idx = block_reduce(idx, OpMinI(), 0x7fffffff, iscratch);
    if (tid == 0) *dst = idx;
    if (a.probs_out != nullptr) {
#pragma unroll
      for (int i = 0; i < SMP_IPT; ++i)
        if (i < ipt && base + i < V) a.probs_out[static_cast<size_t>(r) * V + base + i] = (base + i == idx) ? 1.f : 0.f;
    }
    return;
  }

  // ---- top-k: threshold = k-th largest value, ties kept (sampling.py:17-18) ----
  // 32-step bitwise bisection on the order-preserving integer image of the logits.  The image is computed ONCE (it lives in
  // z's registers for the duration of the search) and a step costs 32 compares, one redux.sync, one shared-memory atomic per
  // warp and ONE __syncthreads (three rotating counters): the first version re-derived the image in every step and paid a
  // three-barrier, two-level shuffle reduction per step - 58 us per launch at top-k 2048 (profiles/r2_configs_final.txt).
  if (top_k > 0 && top_k < V) {
    __shared__ int cnt3[3];
    const int lane = tid & 31;
#pragma unroll
    for (int i = 0; i < SMP_IPT; ++i) z[i] = __uint_as_float(float_order_key(z[i]));
    if (tid < 3) cnt3[tid] = 0;
    __syncthreads();
    uint32_t thr = 0;
    int buf = 0;
    for (int bit = 31; bit >= 0; --bit) {
      const uint32_t cand = thr | (1u << bit);
      int cnt = 0;
#pragma unroll
      for (int i = 0; i < SMP_IPT; ++i) cnt += (__float_as_uint(z[i]) >= cand) ? 1 : 0;
      cnt = __reduce_add_sync(0xffffffffu, cnt);
      if (lane == 0) atomicAdd(&cnt3[buf], cnt);
      __syncthreads();
      const int total = cnt3[buf];
      // the counter of the step before this one was last read before this step's barrier and is next added to after the
      // next step's barrier: thread 0 clears it in between
      const int prev = buf == 0 ? 2 : buf - 1;
      if (tid == 0) cnt3[prev] = 0;
      buf = buf == 2 ? 0 : buf + 1;
      if (total >= top_k) thr = cand;
    }
#pragma unroll
    for (int i = 0; i < SMP_IPT; ++i) {
      const uint32_t k = __float_as_uint(z[i]);
      // back from the image: keys with the top bit set were non-negative floats (bit flipped), the others negative (all flipped)
      z[i] = (k < thr) ? -INFINITY : __uint_as_float((k & 0x80000000u) ? (k ^ 0x80000000u) : ~k);
    }
  }

  // ---- softmax (F.softmax, hierarchical_ar.py:765), in place: z[] becomes the probabilities ----
  float lsum = 0.f;
#pragma unroll
  for (int i = 0; i < SMP_IPT; ++i) {
    z[i] = (z[i] == -INFINITY) ? 0.f : expf(z[i] - mx);
    lsum += z[i];
  }
  const float Z = block_reduce(lsum, OpSumF(), 0.f, fscratch);
  const float invZ = 1.0f / Z;
#pragma unroll
  for (int i = 0; i < SMP_IPT; ++i) z[i] *= invZ;
  float (&wgt)[SMP_IPT] = z;

  // ---- top-p (sampling.py:22-37): keep the smallest upper set {p_i >= c*} whose mass reaches p; among
  //      entries equal to c* keep, in index order, those whose preceding cumulative mass is still < p ----
  if (top_p > 0.f && top_p < 1.f) {
    // 31-step bisection on the kept mass: per step a warp shuffle tree, one partial per warp into a double-buffered array,
    // ONE __syncthreads, and every thread adds the partials in warp order (fixed order: deterministic)
    __shared__ float part2[2][32];
    const int lane_p = tid & 31, w_p = tid >> 5, nw_p = nthr >> 5;
    uint32_t cstar = 0;
    int pbuf = 0;
    for (int bit = 30; bit >= 0; --bit) {   // probabilities are non-negative: sign bit never set
      const uint32_t cand = cstar | (1u << bit);
      float mass = 0.f;
#pragma unroll
      for (int i = 0; i < SMP_IPT; ++i) mass += (__float_as_uint(wgt[i]) >= cand) ? wgt[i] : 0.f;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) mass += __shfl_xor_sync(0xffffffffu, mass, o);
      if (lane_p == 0) part2[pbuf][w_p] = mass;
      __syncthreads();
      float tot = 0.f;
      for (int k2 = 0; k2 < nw_p; ++k2) tot += part2[pbuf][k2];
      pbuf ^= 1;
      if (tot >= top_p) cstar = cand;
    }
    float above = 0.f;
    int ties = 0;
#pragma unroll
    for (int i = 0; i < SMP_IPT; ++i) {
      const uint32_t u = __float_as_uint(wgt[i]);
      above += (u > cstar) ? wgt[i] : 0.f;
      ties += (u == cstar && wgt[i] > 0.f) ? 1 : 0;
    }
    above = block_reduce(above, OpSumF(), 0.f, fscratch);
    const int n_ties = block_reduce(ties, OpSumI(), 0, iscratch);
    const float vstar = __uint_as_float(cstar);
    int keep_ties = 0;   // number of boundary-valued entries whose preceding mass above + m * v* is < p
    {
      float cum = above;
      while (keep_ties < n_ties && cum < top_p) { ++keep_ties; cum += vstar; }
      if (keep_ties == 0) keep_ties = 1;   // the first sorted entry is always kept
    }
    // exclusive prefix of tie counts across threads (only matters when some ties are cut)
    int tie_before = 0;
    if (keep_ties < n_ties) {
      const int lane = tid & 31, w = tid >> 5, nw = nthr >> 5;
      int incl = ties;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int n = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += n;
      }
      __syncthreads();
      if (lane == 31) iscratch[w] = incl;
      __syncthreads();
      int woff = 0;
      for (int k2 = 0; k2 < w && k2 < nw; ++k2) woff += iscratch[k2];
      tie_before = woff + incl - ties;
      __syncthreads();
    }
    float ksum = 0.f;
#pragma unroll
    for (int i = 0; i < SMP_IPT; ++i) {
      const uint32_t u = __float_as_uint(wgt[i]);
      bool keep = u > cstar;
      if (u == cstar && wgt[i] > 0.f) { keep = tie_before < keep_ties; ++tie_before; }
      if (!keep) wgt[i] = 0.f;
      ksum += wgt[i];
    }
    ksum = block_reduce(ksum, OpSumF(), 0.f, fscratch);
    const float inv = 1.0f / ksum;
#pragma unroll
    for (int i = 0; i < SMP_IPT; ++i) wgt[i] *= inv;   // renormalise (sampling.py:36)
  }
  if (a.probs_out != nullptr) {
#pragma unroll
    for (int i = 0; i < SMP_IPT; ++i)
      if (i < ipt && base + i < V) a.probs_out[static_cast<size_t>(r) * V + base + i] = wgt[i];
  }

  // ---- categorical draw: inverse CDF in index order, one Philox uniform per row ----
  float local = 0.f;
#pragma unroll
  for (int i = 0; i < SMP_IPT; ++i) local += wgt[i];
  float excl, total;
  {
    const int lane = tid & 31, w = tid >> 5, nw = nthr >> 5;
    float incl = local;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const float n = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += n;
    }
    __syncthreads();
    if (lane == 31) wsum[w] = incl;
    __syncthreads();
    float woff = 0.f, tot = 0.f;
    for (int k2 = 0; k2 < nw; ++k2) {
      if (k2 < w) woff += wsum[k2];
      tot += wsum[k2];
    }
    float prev = __shfl_up_sync(0xffffffffu, incl, 1);
    if (lane == 0) prev = 0.f;
    excl = woff + prev;
    total = tot;
  }
  const uint64_t grow = row_offset + static_cast<uint64_t>(b);
  uint32_t rnd[4];
  philox4x32_10(static_cast<uint32_t>(seed), static_cast<uint32_t>(seed >> 32), static_cast<uint32_t>(grow),
                static_cast<uint32_t>(grow >> 32), static_cast<uint32_t>(a.pos), static_cast<uint32_t>(slot), rnd);
  const float target = u01_from_bits(rnd[0]) * total;
  int cand = -1;
  float run = excl;
#pragma unroll
  for (int i = 0; i < SMP_IPT; ++i) {
    if (wgt[i] > 0.f && run <= target) cand = base + i;
    run += wgt[i];
  }
  cand = block_reduce(cand, OpMaxI(), -1, iscratch);
  if (tid == 0) *dst = cand;
}

// Stage 2 of the fused head + sampler (gemm.cuh: epilogue_sample_tile): one warp per logits row draws the 32-column chunk
// from softmax(L_chunk) by inverse CDF in chunk order and emits that chunk's pre-drawn index.  `part`: [R, n_chunks]
// (log-sum-exp, index bits).  Destination logic as in sample_kernel.
constexpr int SMPF_WARPS = 8;
__global__ void __launch_bounds__(SMPF_WARPS * 32) sample_finalize_kernel(int trace_id, SampleArgs a, const float2* __restrict__ part,
                                                                          int n_chunks) {
  TraceScope trace_scope(trace_id);
  pdl_launch_dependents();
  pdl_wait();
  const int lane = threadIdx.x & 31;
  const int r = blockIdx.x * SMPF_WARPS + (threadIdx.x >> 5);
  if (r >= a.R) return;
  const int b = r / a.rows_per_b, jj = r % a.rows_per_b;
  const int slot = a.slot0 + jj;
  const float2* p = part + static_cast<size_t>(r) * n_chunks;
  const int per = (n_chunks + 31) / 32;                         // contiguous chunks per lane: prefix order == index order
  const int c0 = lane * per, c1 = min(n_chunks, c0 + per);
  float mx = -INFINITY;
  for (int c = c0; c < c1; ++c) mx = fmaxf(mx, p[c].x);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  float local = 0.f;
  for (int c = c0; c < c1; ++c) local += expf(p[c].x - mx);
  float incl = local;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const float n = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += n;
  }
  const float total = __shfl_sync(0xffffffffu, incl, 31);
  const uint64_t seed = a.sp->seed, grow = a.sp->row_offset + static_cast<uint64_t>(b);
  uint32_t rnd[4];
  philox4x32_10(static_cast<uint32_t>(seed), static_cast<uint32_t>(seed >> 32), static_cast<uint32_t>(grow),
                static_cast<uint32_t>(grow >> 32), static_cast<uint32_t>(a.pos), static_cast<uint32_t>(slot) | 0x100u, rnd);
  const float target = u01_from_bits(rnd[0]) * total;
  int cand = -1;
  float run = incl - local;
  for (int c = c0; c < c1; ++c) {
    const float w = expf(p[c].x - mx);
    if (w > 0.f && run <= target) cand = c;
    run += w;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) cand = max(cand, __shfl_xor_sync(0xffffffffu, cand, o));
  if (lane == 0) {
    int64_t* dst = a.dst_codes + (static_cast<size_t>(b) * a.S + a.pos) * a.dst_w +
                   (a.rows_per_b == 1 ? (a.bot_slot < 0 ? 0 : a.bot_slot) : jj);
    *dst = static_cast<int64_t>(__float_as_int(p[cand < 0 ? 0 : cand].y));
  }
}

}  // namespace hq
