// Host side of the stage-1 decoder (included at the end of engine.cu): context, parameter registry by the reference's
// state_dict names (hqvae/models/stage1/generator.py:243-250, stage1/modules/layers.py:77-186, 300-383), the layer sequence
// of `decode_code`, and the hq_s1_* entry points of include/hqgraft.h.
#pragma once

#include "stage1.cuh"

struct S1Conv {
  int Cin = 0, Cout = 0, CoutPad = 0, taps = 1, bn = 0;
  void* w = nullptr;        // [CoutPad, taps * Cin] tap-major operand type (bf16 | fp32 rounded to TF32), rows >= Cout zero
  float* bias = nullptr;    // [CoutPad]
  CUtensorMap wmap;         // box {one 128-byte row: 64 bf16 | 32 fp32, bn / 2}
};
struct S1Norm { int C = 0; float* g = nullptr; float* b = nullptr; };
struct S1Res { S1Norm n1, n2; S1Conv c1, c2, nin; bool has_nin = false; };
struct S1Attn { S1Norm n; S1Conv qkv, proj; };
struct S1Level { std::vector<S1Res> blocks; std::vector<S1Attn> attns; bool has_attn = false; S1Conv up; int res = 0; };

struct S1Slot {
  int kind = 0;             // 0: fp32 copy, 1: conv weight (packed into `conv` at row `row_off`)
  float* dst = nullptr;
  S1Conv* conv = nullptr;
  int row_off = 0;
  std::vector<int64_t> shape;
  bool loaded = false, ignored = false;
};

struct hq_s1_ctx {
  hq_s1_config cfg;
  int prec = HQ_PREC_BF16;          // HQ_PREC_BF16 | HQ_PREC_TF32: operand type of the convolutions (stage1.cuh)
  size_t esz = 2;                   // its bytes
  int device = 0, max_batch = 0;
  std::string err;
  PFN_encodeTiled encode = nullptr;
  int num_sms = 0;
  float *E_t = nullptr, *E_b = nullptr;
  S1Conv post_quant, conv_in, conv_out;
  S1Res mid1, mid2;
  S1Attn mid_attn;
  std::vector<S1Level> levels;          // lowest resolution first
  S1Norm norm_out;
  std::map<std::string, S1Slot> params;
  float *X = nullptr, *T = nullptr, *S = nullptr;
  void *H = nullptr, *H2 = nullptr, *QKV = nullptr;   // operand type
  double* gn_part = nullptr;      // [B][32 groups][<= 64 row slices][sum, sum of squares]
  float2* gn_stat = nullptr;      // [B][32] (mean, rstd) published by the last slice CTA
  unsigned* gn_cnt = nullptr;     // [B] ticket counters (wrap to 0)
  size_t act_elems = 0;                 // elements of X / T / S / H / H2 per buffer
  size_t device_bytes = 0;
  std::vector<void*> allocs;
  cudaError_t launch_err = cudaSuccess;
  int64_t conv_launches = 0;
  double conv_flops = 0.0;              // of the last decode
};

static void s1_err(hq_s1_ctx* ctx, const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  g_last_error = buf;
  if (ctx) ctx->err = buf;
}
#define S1_CUDA(ctx, call)                                                                       \
  do {                                                                                           \
    cudaError_t e__ = (call);                                                                    \
    if (e__ != cudaSuccess) {                                                                    \
      s1_err(ctx, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__), __FILE__, __LINE__);  \
      return HQ_ERR_CUDA;                                                                        \
    }                                                                                            \
  } while (0)

static int s1_alloc(hq_s1_ctx* ctx, void** p, size_t bytes) {
  bytes = (bytes + 255) & ~static_cast<size_t>(255);
  S1_CUDA(ctx, cudaMalloc(p, bytes));
  S1_CUDA(ctx, cudaMemset(*p, 0, bytes));
  ctx->allocs.push_back(*p);
  ctx->device_bytes += bytes;
  return HQ_OK;
}

// a [rows, cols] matrix of the ctx's operand type, boxes of one 128-byte swizzled row (64 bf16 | 32 fp32) x box_rows
static int s1_map(hq_s1_ctx* ctx, CUtensorMap* m, const void* base, uint64_t rows, uint64_t cols, uint32_t box_rows) {
  const bool f32 = ctx->prec == HQ_PREC_TF32;
  cuuint64_t dims[2] = {cols, rows};
  cuuint64_t strides[1] = {cols * ctx->esz};
  cuuint32_t box[2] = {static_cast<cuuint32_t>(128 / ctx->esz), box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = ctx->encode(m, f32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
                           CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                           CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    s1_err(ctx, "cuTensorMapEncodeTiled failed (%d) rows=%llu cols=%llu box_rows=%u", static_cast<int>(r),
           static_cast<unsigned long long>(rows), static_cast<unsigned long long>(cols), box_rows);
    return HQ_ERR_CUDA;
  }
  return HQ_OK;
}

static void s1_reg(hq_s1_ctx* ctx, const std::string& name, int kind, float* dst, S1Conv* conv, int row_off,
                   std::vector<int64_t> shape) {
  S1Slot s;
  s.kind = kind; s.dst = dst; s.conv = conv; s.row_off = row_off; s.shape = shape;
  ctx->params[name] = s;
}

// a convolution `name` ([Cout, Cin, k, k] + bias); `fused`: extra names whose rows follow (q | k | v as one [3C, C] GEMM).
// bn: tile width; 0 = the planner's choice (Cout rounded up to 32, at most 256)
static int s1_make_conv(hq_s1_ctx* ctx, S1Conv* c, const std::vector<std::string>& names, int Cin, int Cout_each, int k,
                        int bn = 0) {
  const int n = static_cast<int>(names.size());
  c->Cin = Cin;
  c->Cout = Cout_each * n;
  c->taps = k * k;
  if (Cin % 64 != 0) {
    s1_err(ctx, "stage-1 convolution %s: %d input channels (must be a multiple of 64)", names[0].c_str(), Cin);
    return HQ_ERR_UNSUPPORTED;
  }
  if (bn == 0) {
    bn = (c->Cout + 31) / 32 * 32;
    if (bn > 256) bn = 256;
  }
  c->bn = bn;
  c->CoutPad = (c->Cout + bn - 1) / bn * bn;
  int rc;
  if ((rc = s1_alloc(ctx, reinterpret_cast<void**>(&c->w), static_cast<size_t>(c->CoutPad) * c->taps * Cin * ctx->esz))) return rc;
  if ((rc = s1_alloc(ctx, reinterpret_cast<void**>(&c->bias), static_cast<size_t>(c->CoutPad) * 4))) return rc;
  if ((rc = s1_map(ctx, &c->wmap, c->w, c->CoutPad, static_cast<uint64_t>(c->taps) * Cin, static_cast<uint32_t>(bn / 2)))) return rc;
  for (int i = 0; i < n; ++i) {
    s1_reg(ctx, names[i] + ".weight", 1, nullptr, c, i * Cout_each, {Cout_each, Cin, k, k});
    s1_reg(ctx, names[i] + ".bias", 0, c->bias + i * Cout_each, nullptr, 0, {Cout_each});
  }
  return HQ_OK;
}
static int s1_make_norm(hq_s1_ctx* ctx, S1Norm* n, const std::string& name, int C) {
  n->C = C;
  if (C % 32 != 0 || C > 1024) {
    s1_err(ctx, "GroupNorm(32) over %d channels (multiple of 32, <= 1024)", C);
    return HQ_ERR_UNSUPPORTED;
  }
  int rc;
  if ((rc = s1_alloc(ctx, reinterpret_cast<void**>(&n->g), static_cast<size_t>(C) * 4))) return rc;
  if ((rc = s1_alloc(ctx, reinterpret_cast<void**>(&n->b), static_cast<size_t>(C) * 4))) return rc;
  s1_reg(ctx, name + ".weight", 0, n->g, nullptr, 0, {C});
  s1_reg(ctx, name + ".bias", 0, n->b, nullptr, 0, {C});
  return HQ_OK;
}
static int s1_make_res(hq_s1_ctx* ctx, S1Res* r, const std::string& p, int cin, int cout) {
  int rc;
  if ((rc = s1_make_norm(ctx, &r->n1, p + ".norm1", cin))) return rc;
  if ((rc = s1_make_conv(ctx, &r->c1, {p + ".conv1"}, cin, cout, 3))) return rc;
  if ((rc = s1_make_norm(ctx, &r->n2, p + ".norm2", cout))) return rc;
  if ((rc = s1_make_conv(ctx, &r->c2, {p + ".conv2"}, cout, cout, 3))) return rc;
  r->has_nin = cin != cout;
  if (r->has_nin && (rc = s1_make_conv(ctx, &r->nin, {p + ".nin_shortcut"}, cin, cout, 1))) return rc;
  return HQ_OK;
}
static int s1_make_attn(hq_s1_ctx* ctx, S1Attn* a, const std::string& p, int c) {
  int rc;
  if ((rc = s1_make_norm(ctx, &a->n, p + ".norm", c))) return rc;
  if ((rc = s1_make_conv(ctx, &a->qkv, {p + ".q", p + ".k", p + ".v"}, c, c, 1))) return rc;
  return s1_make_conv(ctx, &a->proj, {p + ".proj_out"}, c, c, 1);
}

// device, tensor-map encoder and kernel attributes of a ctx whose precision is set
static int s1_open(hq_s1_ctx* ctx, int device) {
  int rc;
  if (ctx->prec != HQ_PREC_BF16 && ctx->prec != HQ_PREC_TF32) {
    s1_err(ctx, "stage-1 precision %d: HQ_PREC_BF16 (0) or HQ_PREC_TF32 (3)", ctx->prec);
    return HQ_ERR_INVALID;
  }
  ctx->esz = ctx->prec == HQ_PREC_TF32 ? 4 : 2;
  ctx->device = device;
  {
    hq_ctx tmp;
    if ((rc = check_device(&tmp, device))) { s1_err(ctx, "%s", tmp.err.c_str()); return rc; }
    S1_CUDA(ctx, cudaSetDevice(device));
    if ((rc = get_encode_fn(&tmp, &ctx->encode))) { s1_err(ctx, "%s", tmp.err.c_str()); return rc; }
  }
  S1_CUDA(ctx, cudaDeviceGetAttribute(&ctx->num_sms, cudaDevAttrMultiProcessorCount, device));
  S1_CUDA(ctx, cudaFuncSetAttribute(conv_tc2_kernel<bf16>, cudaFuncAttributeMaxDynamicSharedMemorySize, CH_SMEM_BYTES));
  S1_CUDA(ctx, cudaFuncSetAttribute(conv_tc2_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, CH_SMEM_BYTES));
  S1_CUDA(ctx, cudaFuncSetAttribute(s1_attn_kernel<bf16>, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024));
  S1_CUDA(ctx, cudaFuncSetAttribute(s1_attn_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024));
  S1_CUDA(ctx, cudaFuncSetAttribute(s1_attn_mma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
  return HQ_OK;
}

static int s1_create_impl(hq_s1_ctx* ctx, const hq_s1_config* cfg, int device, int max_batch) {
  int rc;
  ctx->cfg = *cfg;
  ctx->prec = cfg->precision;
  ctx->max_batch = max_batch;
  if ((rc = s1_open(ctx, device))) return rc;
  const int L = cfg->n_levels, E = cfg->embed_dim;
  if (L < 1 || L > 8 || max_batch < 1 || cfg->resolution % (1 << L) != 0 || E % 64 != 0 || cfg->out_ch < 1 || cfg->out_ch > 32) {
    s1_err(ctx, "unsupported stage-1 configuration");
    return HQ_ERR_UNSUPPORTED;
  }
  const int lat = cfg->resolution >> L;                       // use_init_downsample: True (layers.py:331-332)
  if (lat < 2 || lat % 2 != 0) {
    s1_err(ctx, "latent resolution %d must be even (2 x 2 bottom cells per top code)", lat);
    return HQ_ERR_UNSUPPORTED;
  }
  if ((rc = s1_alloc(ctx, reinterpret_cast<void**>(&ctx->E_t), static_cast<size_t>(cfg->n_embed) * 4 * E * 4))) return rc;
  if ((rc = s1_alloc(ctx, reinterpret_cast<void**>(&ctx->E_b), static_cast<size_t>(cfg->n_embed) * E * 4))) return rc;
  s1_reg(ctx, "quantize_t.embedding", 0, ctx->E_t, nullptr, 0, {cfg->n_embed, 4 * E});
  s1_reg(ctx, "quantize_b.embedding", 0, ctx->E_b, nullptr, 0, {cfg->n_embed, E});
  if ((rc = s1_make_conv(ctx, &ctx->post_quant, {"post_quant_conv_b"}, 2 * E, cfg->z_channels, 1))) return rc;
  const int top = cfg->ch * cfg->ch_mult[L - 1];
  if ((rc = s1_make_conv(ctx, &ctx->conv_in, {"decoder.conv_in"}, cfg->z_channels, top, 3))) return rc;
  if ((rc = s1_make_res(ctx, &ctx->mid1, "decoder.mid.block_1", top, top))) return rc;
  if ((rc = s1_make_attn(ctx, &ctx->mid_attn, "decoder.mid.attn_1", top))) return rc;
  if ((rc = s1_make_res(ctx, &ctx->mid2, "decoder.mid.block_2", top, top))) return rc;
  // activation buffer size: max over the layer sequence of (padded positions per image) x channels
  size_t per_img = static_cast<size_t>(lat + 2) * (lat + 2) * std::max(std::max(2 * E, cfg->z_channels), top);
  int block_in = top, res = lat;
  ctx->levels.resize(L);
  for (int i = 0; i < L; ++i) {
    const int lvl = L - 1 - i;
    S1Level& lv = ctx->levels[i];
    const int block_out = cfg->ch * cfg->ch_mult[lvl];
    lv.res = res;
    lv.has_attn = res == cfg->attn_resolution;
    lv.blocks.resize(cfg->num_res_blocks + 1);
    if (lv.has_attn) lv.attns.resize(cfg->num_res_blocks + 1);
    for (int j = 0; j <= cfg->num_res_blocks; ++j) {
      const std::string p = "decoder.up." + std::to_string(lvl) + ".block." + std::to_string(j);
      per_img = std::max(per_img, static_cast<size_t>(res + 2) * (res + 2) * std::max(block_in, block_out));
      if ((rc = s1_make_res(ctx, &lv.blocks[j], p, block_in, block_out))) return rc;
      block_in = block_out;
      if (lv.has_attn &&
          (rc = s1_make_attn(ctx, &lv.attns[j], "decoder.up." + std::to_string(lvl) + ".attn." + std::to_string(j), block_in)))
        return rc;
    }
    if ((rc = s1_make_conv(ctx, &lv.up, {"decoder.up." + std::to_string(lvl) + ".upsample.conv"}, block_in, block_in, 3))) return rc;
    res *= 2;
    per_img = std::max(per_img, static_cast<size_t>(res + 2) * (res + 2) * block_in);
  }
  if ((rc = s1_make_norm(ctx, &ctx->norm_out, "decoder.norm_out", block_in))) return rc;
  if ((rc = s1_make_conv(ctx, &ctx->conv_out, {"decoder.conv_out"}, block_in, cfg->out_ch, 3))) return rc;
  ctx->act_elems = per_img * max_batch;
  if ((rc = s1_alloc(ctx, reinterpret_cast<void**>(&ctx->X), ctx->act_elems * 4))) return rc;
  if ((rc = s1_alloc(ctx, reinterpret_cast<void**>(&ctx->T), ctx->act_elems * 4))) return rc;
  if ((rc = s1_alloc(ctx, reinterpret_cast<void**>(&ctx->S), ctx->act_elems * 4))) return rc;
  if ((rc = s1_alloc(ctx, &ctx->H, ctx->act_elems * ctx->esz))) return rc;
  if ((rc = s1_alloc(ctx, &ctx->H2, ctx->act_elems * ctx->esz))) return rc;
  const int att_res = cfg->attn_resolution > 0 ? cfg->attn_resolution : lat;
  if ((rc = s1_alloc(ctx, &ctx->QKV, static_cast<size_t>(max_batch) * (att_res + 2) * (att_res + 2) * 3 * top * ctx->esz)))
    return rc;
  if ((rc = s1_alloc(ctx, reinterpret_cast<void**>(&ctx->gn_part), static_cast<size_t>(max_batch) * 32 * 64 * 2 * 8))) return rc;
  if ((rc = s1_alloc(ctx, reinterpret_cast<void**>(&ctx->gn_stat), static_cast<size_t>(max_batch) * 32 * 8))) return rc;
  if ((rc = s1_alloc(ctx, reinterpret_cast<void**>(&ctx->gn_cnt), static_cast<size_t>(max_batch) * 4))) return rc;
  return HQ_OK;
}

extern "C" int hq_s1_create(const hq_s1_config* cfg, int device, int max_batch, hq_s1_ctx** out) {
  if (!cfg || !out) {
    s1_err(nullptr, "hq_s1_create: null argument");
    return HQ_ERR_INVALID;
  }
  *out = nullptr;
  hq_s1_ctx* ctx = new hq_s1_ctx();
  int rc = s1_create_impl(ctx, cfg, device, max_batch);
  if (rc != HQ_OK) {
    g_last_error = ctx->err;
    for (void* p : ctx->allocs) cudaFree(p);
    delete ctx;
    return rc;
  }
  *out = ctx;
  return HQ_OK;
}

extern "C" int hq_s1_destroy(hq_s1_ctx* ctx) {
  if (!ctx) return HQ_OK;
  cudaSetDevice(ctx->device);
  cudaDeviceSynchronize();
  for (void* p : ctx->allocs) cudaFree(p);
  delete ctx;
  return HQ_OK;
}

extern "C" const char* hq_s1_last_error(const hq_s1_ctx* ctx) { return ctx ? ctx->err.c_str() : g_last_error.c_str(); }
extern "C" size_t hq_s1_device_bytes(const hq_s1_ctx* ctx) { return ctx ? ctx->device_bytes : 0; }
extern "C" double hq_s1_last_conv_flops(const hq_s1_ctx* ctx) { return ctx ? ctx->conv_flops : 0.0; }

extern "C" int hq_s1_load_param(hq_s1_ctx* ctx, const char* name, const void* data, int dtype, const int64_t* shape, int ndim,
                                int is_device) {
  if (!ctx || !name || !data || !shape) return HQ_ERR_INVALID;
  S1_CUDA(ctx, cudaSetDevice(ctx->device));
  auto it = ctx->params.find(name);
  if (it == ctx->params.end()) {
    s1_err(ctx, "unexpected key in state_dict: \"%s\"", name);
    return HQ_ERR_INVALID;
  }
  S1Slot& s = it->second;
  bool ok = static_cast<size_t>(ndim) == s.shape.size();
  for (int i = 0; ok && i < ndim; ++i) ok = shape[i] == s.shape[i];
  if (!ok || dtype < HQ_F32 || dtype > HQ_F16) {
    s1_err(ctx, "size / dtype mismatch for %s", name);
    return HQ_ERR_INVALID;
  }
  size_t n = 1;
  for (auto v : s.shape) n *= static_cast<size_t>(v);
  const size_t esz = dtype == HQ_F32 ? 4 : 2;
  void* staged = nullptr;
  const void* src = data;
  if (!is_device) {
    S1_CUDA(ctx, cudaMalloc(&staged, n * esz));
    cudaError_t e = cudaMemcpy(staged, data, n * esz, cudaMemcpyHostToDevice);
    if (e != cudaSuccess) {
      cudaFree(staged);
      s1_err(ctx, "cudaMemcpy H2D failed for %s", name);
      return HQ_ERR_CUDA;
    }
    src = staged;
  }
  float* f32 = s.dst;
  float* tmp = nullptr;
  if (s.kind == 1) {
    if (cudaMalloc(reinterpret_cast<void**>(&tmp), n * 4) != cudaSuccess) {
      if (staged) cudaFree(staged);
      s1_err(ctx, "out of memory loading %s", name);
      return HQ_ERR_CUDA;
    }
    f32 = tmp;
  }
  if (dtype == HQ_F32) launch_convert<float>(src, f32, HQ_PREC_FP32, n);
  else if (dtype == HQ_BF16) launch_convert<bf16>(src, f32, HQ_PREC_FP32, n);
  else launch_convert<__half>(src, f32, HQ_PREC_FP32, n);
  if (s.kind == 1) {
    S1Conv* c = s.conv;
    const size_t off = static_cast<size_t>(s.row_off) * c->taps * c->Cin;
    const int grid = static_cast<int>((n + 255) / 256 > 4096 ? 4096 : (n + 255) / 256);
    if (ctx->prec == HQ_PREC_TF32)
      s1_pack_weight_kernel<float><<<grid, 256>>>(tmp, static_cast<float*>(c->w) + off, static_cast<int>(s.shape[0]), c->Cin, c->taps);
    else
      s1_pack_weight_kernel<bf16><<<grid, 256>>>(tmp, static_cast<bf16*>(c->w) + off, static_cast<int>(s.shape[0]), c->Cin, c->taps);
  }
  cudaError_t e = cudaDeviceSynchronize();
  if (tmp) cudaFree(tmp);
  if (staged) cudaFree(staged);
  if (e != cudaSuccess) {
    s1_err(ctx, "parameter conversion failed for %s: %s", name, cudaGetErrorString(e));
    return HQ_ERR_CUDA;
  }
  s.loaded = true;
  return HQ_OK;
}

extern "C" int hq_s1_params_complete(hq_s1_ctx* ctx) {
  if (!ctx) return HQ_ERR_INVALID;
  std::string missing;
  int n = 0;
  for (auto& kv : ctx->params)
    if (!kv.second.loaded) {
      if (n < 8) missing += (n ? ", " : "") + kv.first;
      ++n;
    }
  if (n) {
    s1_err(ctx, "missing %d stage-1 key(s): %s%s", n, missing.c_str(), n > 8 ? ", ..." : "");
    return HQ_ERR_STATE;
  }
  return HQ_OK;
}

// ---- layer launches (T: the operand type, bf16 or float; see stage1.cuh) ----
static void s1_check(hq_s1_ctx* ctx) {
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess && ctx->launch_err == cudaSuccess) ctx->launch_err = e;
}

template <typename T>
static void s1_conv(hq_s1_ctx* ctx, cudaStream_t st, const S1Conv& c, const void* A, int B, int res, int mode, float* outf,
                    void* outb, const float* resid) {
  const int Hp = res + 2;
  ConvParams p;
  memset(&p, 0, sizeof(p));
  p.R = B * Hp * Hp;
  p.Cin = c.Cin; p.CoutPad = c.CoutPad; p.cout = c.Cout; p.taps = c.taps; p.Hp = Hp; p.Wp = Hp; p.bn = c.bn;
  p.mode = mode; p.ldo = c.Cout; p.bias = c.bias; p.res = resid; p.outf = outf; p.outb = outb;
  CUtensorMap mA;
  if (s1_map(ctx, &mA, A, static_cast<uint64_t>(p.R), static_cast<uint64_t>(c.Cin), 128) != HQ_OK) {
    if (ctx->launch_err == cudaSuccess) ctx->launch_err = cudaErrorInvalidValue;
    return;
  }
  const int tiles = (c.CoutPad / c.bn) * ((p.R + 255) / 256);
  const int pairs = tiles < ctx->num_sms / 2 ? tiles : ctx->num_sms / 2;
  conv_tc2_kernel<T><<<dim3(2 * pairs), dim3(CH_THREADS), CH_SMEM_BYTES, st>>>(mA, c.wmap, p);
  s1_check(ctx);
  ++ctx->conv_launches;
  ctx->conv_flops += 2.0 * B * res * res * static_cast<double>(c.Cout) * c.Cin * c.taps;
}

template <typename T>
static void s1_gn(hq_s1_ctx* ctx, cudaStream_t st, const S1Norm& n, const float* x, void* out, int B, int res, int swish) {
  const int Hp = res + 2;
  const int S = res < 64 ? res : 64;
  s1_gn_stats_kernel<<<dim3(S, B), 256, 0, st>>>(x, ctx->gn_part, ctx->gn_stat, ctx->gn_cnt, Hp, Hp, n.C, S);
  s1_gn_apply_kernel<T><<<dim3(Hp, B), 256, 0, st>>>(x, ctx->gn_stat, n.g, n.b, static_cast<T*>(out), Hp, Hp, n.C, swish);
  s1_check(ctx);
}

template <typename T>
static void s1_resample(hq_s1_ctx* ctx, cudaStream_t st, const float* x, void* out, int B, int res, int C, int up) {
  s1_resample_kernel<T><<<dim3(up * res + 2, B), 256, 0, st>>>(x, static_cast<T*>(out), res, res, C, up);
  s1_check(ctx);
}

// x (ctx->X) -> ResnetBlock (layers.py:118-135); result in ctx->X
template <typename T>
static void s1_resblock(hq_s1_ctx* ctx, cudaStream_t st, const S1Res& r, int B, int res) {
  s1_gn<T>(ctx, st, r.n1, ctx->X, ctx->H, B, res, 1);
  s1_conv<T>(ctx, st, r.c1, ctx->H, B, res, S1_OUT_F32, ctx->T, nullptr, nullptr);
  s1_gn<T>(ctx, st, r.n2, ctx->T, ctx->H, B, res, 1);
  if (r.has_nin) {
    s1_resample<T>(ctx, st, ctx->X, ctx->H2, B, res, r.nin.Cin, 1);                      // operand copy of x
    s1_conv<T>(ctx, st, r.nin, ctx->H2, B, res, S1_OUT_F32, ctx->S, nullptr, nullptr);   // nin_shortcut(x)
    s1_conv<T>(ctx, st, r.c2, ctx->H, B, res, S1_OUT_F32, ctx->S, nullptr, ctx->S);      // + conv2(h), in place
    std::swap(ctx->X, ctx->S);
  } else {
    s1_conv<T>(ctx, st, r.c2, ctx->H, B, res, S1_OUT_F32, ctx->X, nullptr, ctx->X);      // x + conv2(h), in place
  }
}

// AttnBlock (layers.py:163-186); result in ctx->X.  bf16: tensor-core core where the shape allows; float: the fp32 core.
template <typename T>
static void s1_attnblock(hq_s1_ctx* ctx, cudaStream_t st, const S1Attn& a, int B, int res) {
  const int C = a.n.C;
  s1_gn<T>(ctx, st, a.n, ctx->X, ctx->H, B, res, 0);
  s1_conv<T>(ctx, st, a.qkv, ctx->H, B, res, S1_OUT_ACT, nullptr, ctx->QKV, nullptr);
  const int N = res * res;
  static const bool no_mma = getenv("HQ_DEBUG") != nullptr && getenv("HQ_S1_ATTN_SIMT") != nullptr;
  if (std::is_same<T, bf16>::value && !no_mma && N % 16 == 0 && N <= S1A_NMAX && C % S1A_CB == 0 && C <= S1A_CMAX) {
    // tensor-core path: 64 queries per CTA
    const size_t smem = static_cast<size_t>(s1a_smem_bytes(C));
    s1_attn_mma_kernel<<<dim3((N + S1A_Q - 1) / S1A_Q, B), 128, smem, st>>>(static_cast<const bf16*>(ctx->QKV),
                                                                             static_cast<bf16*>(ctx->H2), res, res, C);
  } else {
    const size_t smem = static_cast<size_t>(S1_ATT_Q) * (C + N) * 4;
    s1_attn_kernel<T><<<dim3((N + S1_ATT_Q - 1) / S1_ATT_Q, B), 256, smem, st>>>(static_cast<const T*>(ctx->QKV),
                                                                                 static_cast<T*>(ctx->H2), res, res, C);
  }
  s1_check(ctx);
  s1_conv<T>(ctx, st, a.proj, ctx->H2, B, res, S1_OUT_F32, ctx->X, nullptr, ctx->X);
}

// the layer sequence of decode_code (generator.py:316-367) in operand type T
template <typename T>
static void s1_decode(hq_s1_ctx* ctx, cudaStream_t st, const int64_t* code_t, const int64_t* code_b, float* out, int B) {
  const hq_s1_config& cfg = ctx->cfg;
  const int lat = cfg.resolution >> cfg.n_levels;
  // codes -> [quant_t (pixel-shuffled) | quant_b] -> post_quant_conv_b -> conv_in
  s1_quant_kernel<T><<<B * (lat + 2) * (lat + 2), 256, 0, st>>>(code_t, code_b, ctx->E_t, ctx->E_b, static_cast<T*>(ctx->H),
                                                                 cfg.embed_dim, lat, cfg.n_embed);
  s1_check(ctx);
  s1_conv<T>(ctx, st, ctx->post_quant, ctx->H, B, lat, S1_OUT_F32, ctx->X, nullptr, nullptr);
  s1_resample<T>(ctx, st, ctx->X, ctx->H, B, lat, cfg.z_channels, 1);
  s1_conv<T>(ctx, st, ctx->conv_in, ctx->H, B, lat, S1_OUT_F32, ctx->T, nullptr, nullptr);
  std::swap(ctx->X, ctx->T);
  s1_resblock<T>(ctx, st, ctx->mid1, B, lat);
  s1_attnblock<T>(ctx, st, ctx->mid_attn, B, lat);
  s1_resblock<T>(ctx, st, ctx->mid2, B, lat);
  int res = lat;
  for (auto& lv : ctx->levels) {
    for (size_t j = 0; j < lv.blocks.size(); ++j) {
      s1_resblock<T>(ctx, st, lv.blocks[j], B, res);
      if (lv.has_attn) s1_attnblock<T>(ctx, st, lv.attns[j], B, res);
    }
    s1_resample<T>(ctx, st, ctx->X, ctx->H, B, res, lv.up.Cin, 2);                      // nearest 2x (layers.py:49-52)
    res *= 2;
    s1_conv<T>(ctx, st, lv.up, ctx->H, B, res, S1_OUT_F32, ctx->T, nullptr, nullptr);
    std::swap(ctx->X, ctx->T);
  }
  s1_gn<T>(ctx, st, ctx->norm_out, ctx->X, ctx->H, B, res, 1);
  s1_conv<T>(ctx, st, ctx->conv_out, ctx->H, B, res, S1_OUT_IMAGE, out, nullptr, nullptr);
}

// `SimRQGAN2Generator.decode_code` (generator.py:323-367) with both grids given; device pointers; asynchronous on `stream`.
extern "C" int hq_s1_decode_codes(hq_s1_ctx* ctx, const int64_t* code_t, const int64_t* code_b, float* out, int B, void* stream) {
  if (!ctx || !code_t || !code_b || !out) return HQ_ERR_INVALID;
  int rc = hq_s1_params_complete(ctx);
  if (rc) return rc;
  if (B < 1 || B > ctx->max_batch) {
    s1_err(ctx, "batch %d outside [1, max_batch=%d]", B, ctx->max_batch);
    return HQ_ERR_INVALID;
  }
  S1_CUDA(ctx, cudaSetDevice(ctx->device));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  ctx->launch_err = cudaSuccess;
  ctx->conv_flops = 0.0;
  if (ctx->prec == HQ_PREC_TF32) s1_decode<float>(ctx, st, code_t, code_b, out, B);
  else s1_decode<bf16>(ctx, st, code_t, code_b, out, B);
  if (ctx->launch_err != cudaSuccess) {
    s1_err(ctx, "stage-1 kernel launch failed: %s", cudaGetErrorString(ctx->launch_err));
    return HQ_ERR_CUDA;
  }
  return HQ_OK;
}

// One convolution through s1_make_conv / hq_s1_load_param / s1_conv on a throw-away ctx (include/hqgraft.h).
extern "C" int hq_debug_s1_conv(int prec, const void* A, const float* weight, const float* bias, int B, int res, int Cin,
                                int Cout, int k, int mode, int tile, const float* resid, void* out, void* stream) {
  if (!A || !weight || !bias || !out || B < 1 || res < 1 || Cout < 1 || (k != 1 && k != 3) || mode < S1_OUT_F32 ||
      mode > S1_OUT_IMAGE || (resid && mode != S1_OUT_F32) || (tile != 0 && (tile % 32 != 0 || tile < 32 || tile > 256))) {
    s1_err(nullptr, "hq_debug_s1_conv: bad argument");
    return HQ_ERR_INVALID;
  }
  hq_s1_ctx ctx;
  ctx.prec = prec;
  int device = 0;
  S1_CUDA(&ctx, cudaGetDevice(&device));
  S1Conv c;
  int rc = s1_open(&ctx, device);
  if (!rc) rc = s1_make_conv(&ctx, &c, {"conv"}, Cin, Cout, k, tile);
  const int64_t wshape[4] = {Cout, Cin, k, k}, bshape[1] = {Cout};
  if (!rc) rc = hq_s1_load_param(&ctx, "conv.weight", weight, HQ_F32, wshape, 4, 1);
  if (!rc) rc = hq_s1_load_param(&ctx, "conv.bias", bias, HQ_F32, bshape, 1, 1);
  if (!rc) {
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    float* outf = mode == S1_OUT_ACT ? nullptr : static_cast<float*>(out);
    void* outb = mode == S1_OUT_ACT ? out : nullptr;
    if (prec == HQ_PREC_TF32) s1_conv<float>(&ctx, st, c, A, B, res, mode, outf, outb, resid);
    else s1_conv<bf16>(&ctx, st, c, A, B, res, mode, outf, outb, resid);
    cudaError_t e = ctx.launch_err != cudaSuccess ? ctx.launch_err : cudaStreamSynchronize(st);
    if (e != cudaSuccess) {
      s1_err(&ctx, "hq_debug_s1_conv: %s", cudaGetErrorString(e));
      rc = HQ_ERR_CUDA;
    }
  }
  for (void* p : ctx.allocs) cudaFree(p);
  if (rc) g_last_error = ctx.err;
  return rc;
}
