// libhqgraft engine: context, parameter registry (reference state_dict names -> engine layout),
// the per-position kernel sequence of the HQ sampling loop, CUDA-graph replay, and the C ABI of
// include/hqgraft.h.
#include <cuda.h>
#include <cuda_runtime.h>

#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <algorithm>
#include <cstring>
#include <map>
#include <string>
#include <tuple>
#include <vector>

#include "../../include/hqgraft.h"
#include "common.cuh"
#include "gemm.cuh"
#include "kernels.cuh"
#include "chain.cuh"

using namespace hq;

// ------------------------------------------------------------------------------------------------
// errors
// ------------------------------------------------------------------------------------------------
static thread_local std::string g_last_error;

struct hq_ctx;
static void set_err(hq_ctx* ctx, const char* fmt, ...);

#define HQ_CUDA(ctx, call)                                                                       \
  do {                                                                                           \
    cudaError_t e__ = (call);                                                                    \
    if (e__ != cudaSuccess) {                                                                    \
      set_err(ctx, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__), __FILE__, __LINE__); \
      return HQ_ERR_CUDA;                                                                        \
    }                                                                                            \
  } while (0)

// ------------------------------------------------------------------------------------------------
// context
// ------------------------------------------------------------------------------------------------
// One tensor map per CTA-pair tile width: each CTA of a pair stages BN/2 weight rows per k-block with ONE TMA
// instruction (a TMA issue costs ~40 ns in the producer thread; 16-row boxes made a 256-wide tile issue-bound).
struct PairMaps {
  CUtensorMap m[6];
  CUtensorMap m3[6];     // the same tiles as 3-D boxes {64, BN/2, 2} over the [K/64][N][64] view (two k-blocks per instruction)
  bool have3 = false;
  static int index(int bn) { return bn == 32 ? 0 : bn == 64 ? 1 : bn == 96 ? 2 : bn == 128 ? 3 : bn == 192 ? 4 : bn == 256 ? 5 : -1; }
  static int width(int i) { static const int w[6] = {32, 64, 96, 128, 192, 256}; return w[i]; }
};

struct Weight {          // a GEMM weight [N, K] in the precision's storage type
  void* ptr = nullptr;
  int N = 0, K = 0;
  CUtensorMap map;       // 2-byte engines only: [N, K], box {64, 64}, SWIZZLE_128B (single-CTA kernel)
  PairMaps mapp;         // 2-byte engines only: box {64, BN/2} per pair-tile width BN (CTA-pair kernel: one load per stage per CTA)
  int map_idx = -1;      // index of mapp.m[0] in the ctx's device tensor-map table (chain kernel)
};
struct ABuf {            // a GEMM A operand buffer [rows_pad, K]
  void* ptr = nullptr;
  int rows = 0, K = 0;
  CUtensorMap map;       // 2-byte engines only: box {64, 128}
  CUtensorMap map3;      // 2-byte engines only, K >= 128: 3-D box {64, 128, 2} over the [K/64][rows][64] view (pair kernel, KS = 2)
  bool have3 = false;
  int map_idx = -1;      // index in the ctx's device tensor-map table (chain kernel)
};
struct BlockW {
  Weight qkv, proj, fc1, fc2;
  float *bqkv, *bproj, *b1, *b2, *ln1g, *ln1b, *ln2g, *ln2b;
};
struct ParamSlot {
  void* dst = nullptr;
  int dst_is_weight = 0;   // 1: stored in the GEMM storage type (bf16 | fp16 | fp32); 0: fp32
  std::vector<int64_t> shape;
  bool loaded = false;
  bool ignored = false;    // accepted for strict loading, never read by the sampler
};

typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

// Experiment / test switches.  They are read from the environment ONCE, when a ctx is created (or a stand-alone debug
// hook is entered), and ONLY when HQ_DEBUG=1 is set: a stray HQ_* variable in a production environment changes nothing.
struct DebugSwitches {
  std::string ablate;          // HQ_ABLATE=tag[,tag...]: drop launches whose tag starts with one of the names (timing only)
  int attn_groups = 0;         // HQ_ATTN_GROUPS: head groups per image of the decode attention
  int attn_no_prefetch = 0;    // HQ_ATTN_NO_PREFETCH: no K/V request ahead of griddepcontrol.wait
  int attn_sleep = 0;          // HQ_ATTN_SLEEP (ns), scalar kernel
  int attn_scalar = 0;         // HQ_ATTN_SCALAR: the scalar bulk-staged kernel (also pinned by hq_debug_attention variant 1)
  int attm_stages = 0;         // HQ_ATTM_STAGES
  int attm_per_sm = 0;         // HQ_ATTM_PER_SM
  int attn_generic = 0;        // HQ_ATTN_GENERIC
  int attn_fewkeys_old = 0;    // HQ_ATTN_FEWKEYS_OLD
  int max_splitk = 0;          // HQ_MAX_SPLITK
  int no_splitk = 0;           // HQ_NO_SPLITK
  int force_splitk = 0;        // HQ_FORCE_SPLITK (tests: pin the split-K factor of the residual GEMMs)
  int trace_pdl = 0;           // HQ_TRACE_PDL: keep PDL on while tracing
  int bench_splits = 0;        // HQ_BENCH_SPLITS (hq_bench_gemm_shape)
  int force_bn = 0;            // hq_debug_gemm: pinned tile width (0 = heuristic, -64 / -128 = single-CTA kernel)
  int no_chain = 0;            // HQ_NO_CHAIN: one kernel per op even where the persistent chain kernel applies
  int chain_min_batch = 0;     // HQ_CHAIN_MIN_BATCH: smallest batch that takes the chain kernel (default 129)
  int chain_no_l2pf = 0;       // HQ_CHAIN_NO_L2PF: chain kernel without the L2 prefetch of later weight tiles
  int gemm_ks1 = 0;            // HQ_GEMM_KS1: pair GEMM with one k-block per ring stage (2-D boxes) everywhere
  int bn_m256 = 0;             // HQ_BN_M256: pinned pair-tile width of the unsplit GEMMs with M <= 256 (plan experiments)
};

static int env_int(const char* name) {
  const char* v = getenv(name);
  return v ? atoi(v) : 0;
}
static DebugSwitches read_debug_switches() {
  DebugSwitches d;
  const char* on = getenv("HQ_DEBUG");
  if (on == nullptr || atoi(on) == 0) return d;
  if (const char* a = getenv("HQ_ABLATE")) d.ablate = a;
  d.attn_groups = env_int("HQ_ATTN_GROUPS");
  d.attn_no_prefetch = getenv("HQ_ATTN_NO_PREFETCH") != nullptr;
  d.attn_sleep = env_int("HQ_ATTN_SLEEP");
  d.attn_scalar = getenv("HQ_ATTN_SCALAR") != nullptr;
  d.attm_stages = env_int("HQ_ATTM_STAGES");
  d.attm_per_sm = env_int("HQ_ATTM_PER_SM");
  d.attn_generic = getenv("HQ_ATTN_GENERIC") != nullptr;
  d.attn_fewkeys_old = getenv("HQ_ATTN_FEWKEYS_OLD") != nullptr;
  d.max_splitk = env_int("HQ_MAX_SPLITK");
  d.no_splitk = getenv("HQ_NO_SPLITK") != nullptr;
  d.force_splitk = env_int("HQ_FORCE_SPLITK");
  d.trace_pdl = getenv("HQ_TRACE_PDL") != nullptr;
  d.bench_splits = env_int("HQ_BENCH_SPLITS");
  d.no_chain = getenv("HQ_NO_CHAIN") != nullptr;
  d.chain_min_batch = env_int("HQ_CHAIN_MIN_BATCH");
  d.chain_no_l2pf = getenv("HQ_CHAIN_NO_L2PF") != nullptr;
  d.gemm_ks1 = getenv("HQ_GEMM_KS1") != nullptr;
  d.bn_m256 = env_int("HQ_BN_M256");
  return d;
}

struct GraphKey {
  int B, S, p0, p1, forced_top, forced_bot, sos_override, tracing, prefix_len;
  bool operator<(const GraphKey& o) const {
    return std::tie(B, S, p0, p1, forced_top, forced_bot, sos_override, tracing, prefix_len) <
           std::tie(o.B, o.S, o.p0, o.p1, o.forced_top, o.forced_bot, o.sos_override, o.tracing, o.prefix_len);
  }
};

struct hq_ctx {
  hq_config cfg;
  int device = 0, max_batch = 0;
  // The 2-byte tensor-core engine (HQ_PREC_BF16 / HQ_PREC_F16): tcgen05 GEMMs, split-K, the mma.sync decode attention,
  // the fused head sampler; false: the fp32 CUDA-core engine.  `prec` names the element type.
  bool half = true;
  int prec = HQ_PREC_BF16;
  int D = 0, nh = 0, L = 0, Ld = 0, Vt = 0, Vb = 0, Vmax = 0, T0 = 1, Tc = 0, Smax = 0;
  size_t wsize = 2;  // bytes per GEMM weight / activation element
  std::string err;
  std::vector<void*> allocs;       // parameters (live as long as the ctx)
  std::vector<void*> act_allocs;   // batch-sized state (re-made by hq_reserve_batch)
  std::vector<void*> pre_allocs;   // image-completion workspace (grown on demand by runs with a prefix, freed with act_allocs)
  bool alloc_act = false, alloc_pre = false;
  size_t device_bytes = 0, act_bytes = 0, pre_bytes = 0;
  std::map<std::string, ParamSlot> params;
  PFN_encodeTiled encode = nullptr;

  std::vector<BlockW> blocks, depths;
  Weight head_top, head_bot;
  float *sos_table = nullptr, *sos_depth = nullptr;
  float *E_top = nullptr, *E_bot = nullptr, *P_emb = nullptr, *P_top = nullptr;
  float *E_txt = nullptr, *P_txt = nullptr;
  float *E_top_depth = nullptr, *P_depth = nullptr;
  float *E_bot_depth = nullptr;                       // 'top2bot' only (tok_emb_bot_depth is unused by 'parallel' sampling)
  float *P_top_h = nullptr, *P_top_w = nullptr;       // position_embedding == '2d'
  int Hpos = 0;                                       // rows of pos_emb_top_h / _w = sqrt(ctx_len_img)
  int depth_rows = 4;                                 // rows per image of the widest depth pass (5: 'bidirectional', 16: 3 levels)
  // 3-level HQTransformer (code_levels == 3): E_top / E_bot / head_top / head_bot / lnt / lnb are levels 0 and 2
  int levels = 2, n_stack = 5, Vm = 0;
  float *E_mid = nullptr, *E_mid_depth = nullptr, *P_depth2 = nullptr, *lnm_g = nullptr, *lnm_b = nullptr;
  Weight head_mid;
  int64_t* codes_mid = nullptr;
  float *lnf_g = nullptr, *lnf_b = nullptr, *lnt_g = nullptr, *lnt_b = nullptr, *lnb_g = nullptr, *lnb_b = nullptr;

  // activations / state
  ABuf h, att, mlp;
  void* q = nullptr;
  float *x = nullptr, *yd = nullptr, *logits = nullptr;
  float2* samp_part = nullptr;     // fused head + sampler: [depth_rows * B, Vmax / 32] (log-sum-exp, drawn index) per 32-column chunk
  float* splitk_ws = nullptr;   // [LN_MAXFOLD][rows][D] fp32 partial sums of split-K fc2 GEMMs (folded in by the next LayerNorm)
  unsigned int* att_sched = nullptr;   // [2] work-ticket / finished-CTA counters of attention_decode_mma_kernel (rest at 0)
  CUtensorMap kmap, vmap;              // spatial KV cache as [rows = L*B*Tc][heads][64] 2-byte, box {64, hpc, 8}, SWIZZLE_128B
  bool kv_maps = false;
  int num_sms = 0;
  int ws_rows = 0;
  // image completion: the causal prefix pass runs on its own activation buffers of pre_rows rows (B x (T0 + P - 1) tokens;
  // swapped in for h / att / mlp / q while it runs), so that a run without a prefix allocates nothing
  ABuf pre_h, pre_att, pre_mlp;
  void* pre_q = nullptr;
  float* pre_x = nullptr;
  int pre_rows = 0;
  bool prefix_pass = false;        // attention(): causal multi-token calls take attention_prefix_kernel (2-byte engines)
  void *kc = nullptr, *vc = nullptr, *kd = nullptr, *vd = nullptr;
  int64_t *cond = nullptr, *codes_top = nullptr, *codes_bot = nullptr;
  float* sos_override = nullptr;
  hq_sampling_params* d_sp = nullptr;

  cudaStream_t own_stream = nullptr;
  struct GraphEntry { cudaGraphExec_t exec; int64_t launches; uint64_t stamp; };
  static constexpr size_t kMaxGraphs = 96;   // LRU-capped: the per-position sampling_step API captures one graph per position
  std::map<GraphKey, GraphEntry> graphs;
  int64_t launches = 0;
  int64_t last_launches = 0;
  cudaError_t launch_err = cudaSuccess;
  bool use_pdl = false;
  bool tracing = false;
  int trace_cap = 0;
  std::vector<std::string> trace_tags;
  bool full_dependency_next = false;   // the next launch is an ordinary (complete-then-start) dependency even under PDL
  std::string tag_suffix;   // shape annotation appended to the next launch tag (tracing only)
  DebugSwitches dbg = read_debug_switches();
  uint64_t graph_clock = 0;   // LRU stamp source of the graph cache

  // ---- persistent op-chain kernel (chain.cuh) ----
  bool chain_ok = false;               // kernel attributes set and enough CTA pairs co-resident
  int chain_grid = 0;                  // CTAs of every chain launch (2 x co-resident pairs)
  CUtensorMap* d_maps = nullptr;       // tensor-map table: A buffers, then six pair maps per weight (rebuilt by reserve)
  ChainOp* d_ops = nullptr;            // arena of op tables, deduplicated by content
  int ops_cap = 0, ops_used = 0;
  std::map<std::string, int> chain_index;   // op-table bytes -> first op in d_ops
  unsigned long long* d_chain_bar = nullptr;
  unsigned long long chain_epoch = 0;  // arrivals of the chain launches enqueued so far in this run
  enum { CHAIN_OFF = 0, CHAIN_PLAN = 1, CHAIN_RUN = 2 };
  int chain_mode = CHAIN_OFF;          // PLAN: build + upload op tables, launch nothing (done before graph capture)
  bool recording = false;              // ops are appended to `rec` instead of being launched
  std::vector<ChainOp> rec;
  std::vector<std::string> rec_tags;
  int rec_flags = 0;                   // flags of the next recorded GEMM op (CH_F_T0_RT)
  const char* gemm_tag_override = nullptr;   // timeline tag of the next GEMM launch (split-K residual GEMMs: "gemm_resid")
  ChainRt chain_rt;                    // t0 / pos / S of the position being recorded
  std::vector<char> trace_chain_cont;  // tracing: entry i is op > 0 of a chain launch (its start is entry i-1's end)
  int64_t chain_launches = 0, chain_ops = 0;
  int chain_launches_run = 0;          // chain launches of the current run (selects the instrumented one)
  int phase_launch = -1, phase_op = -1;   // hq_debug_chain_phases: which launch of the run / which of its ops is stamped
};

static void set_err(hq_ctx* ctx, const char* fmt, ...) {
  char buf[2048];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  g_last_error = buf;
  if (ctx) ctx->err = buf;
}

static int dev_alloc(hq_ctx* ctx, void** p, size_t bytes) {
  bytes = (bytes + 255) & ~static_cast<size_t>(255);
  HQ_CUDA(ctx, cudaMalloc(p, bytes));
  HQ_CUDA(ctx, cudaMemset(*p, 0, bytes));
  if (ctx->alloc_pre) {
    ctx->pre_allocs.push_back(*p);
    ctx->pre_bytes += bytes;
  } else if (ctx->alloc_act) {
    ctx->act_allocs.push_back(*p);
    ctx->act_bytes += bytes;
  } else {
    ctx->allocs.push_back(*p);
    ctx->device_bytes += bytes;
  }
  return HQ_OK;
}

// Element type of the tensor maps of a 2-byte engine (TMA moves the same bytes either way; the map names what the kernels read)
static CUtensorMapDataType tmap_dtype(const hq_ctx* ctx) {
  return ctx->prec == HQ_PREC_F16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;
}

static int make_map(hq_ctx* ctx, CUtensorMap* m, void* base, uint64_t rows, uint64_t cols, uint32_t box_rows) {
  cuuint64_t dims[2] = {cols, rows};
  cuuint64_t strides[1] = {cols * 2};
  cuuint32_t box[2] = {64, box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = ctx->encode(m, tmap_dtype(ctx), 2, base, dims, strides, box, estr,
                           CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                           CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_err(ctx, "cuTensorMapEncodeTiled failed (%d) rows=%llu cols=%llu", static_cast<int>(r),
            static_cast<unsigned long long>(rows), static_cast<unsigned long long>(cols));
    return HQ_ERR_CUDA;
  }
  return HQ_OK;
}

// [rows, cols] 2-byte elements viewed as [cols / 64][rows][64]: one box {64, box_rows, ks} stages ks consecutive 64-wide
// k-blocks of box_rows rows as ks consecutive SWIZZLE_128B tiles (what the UMMA descriptors of ks k-blocks expect)
static int make_map3(hq_ctx* ctx, CUtensorMap* m, void* base, uint64_t rows, uint64_t cols, uint32_t box_rows, uint32_t ks) {
  cuuint64_t dims[3] = {64, rows, cols / 64};
  cuuint64_t strides[2] = {cols * 2, 128};
  cuuint32_t box[3] = {64, box_rows, ks};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = ctx->encode(m, tmap_dtype(ctx), 3, base, dims, strides, box, estr,
                           CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                           CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_err(ctx, "cuTensorMapEncodeTiled (3-D k-block view) failed (%d) rows=%llu cols=%llu box_rows=%u", static_cast<int>(r),
            static_cast<unsigned long long>(rows), static_cast<unsigned long long>(cols), box_rows);
    return HQ_ERR_CUDA;
  }
  return HQ_OK;
}

static int make_pair_maps(hq_ctx* ctx, PairMaps* pm, void* base, uint64_t rows, uint64_t cols) {
  memset(pm, 0, sizeof(*pm));
  pm->have3 = cols >= 128;
  for (int i = 0; i < 6; ++i) {
    if (static_cast<uint64_t>(PairMaps::width(i)) > rows) continue;   // a tile wider than the matrix is never launched
    int rc = make_map(ctx, &pm->m[i], base, rows, cols, static_cast<uint32_t>(PairMaps::width(i) / 2));
    if (rc) return rc;
    if (pm->have3 && (rc = make_map3(ctx, &pm->m3[i], base, rows, cols, static_cast<uint32_t>(PairMaps::width(i) / 2), 2))) return rc;
  }
  return HQ_OK;
}

// KV cache rows as a 3-D tensor {64 dims, n_heads, rows}: one box = 8 cache rows of one head group (hpc heads)
static int make_kv_map(hq_ctx* ctx, CUtensorMap* m, const void* base, int n_heads, uint64_t rows, int hpc) {
  cuuint64_t dims[3] = {64, static_cast<cuuint64_t>(n_heads), rows};
  cuuint64_t strides[2] = {128, static_cast<cuuint64_t>(n_heads) * 128};
  cuuint32_t box[3] = {64, static_cast<cuuint32_t>(hpc), 8};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = ctx->encode(m, tmap_dtype(ctx), 3, const_cast<void*>(base), dims, strides, box, estr,
                           CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                           CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_err(ctx, "cuTensorMapEncodeTiled (KV cache) failed (%d) heads=%d rows=%llu hpc=%d", static_cast<int>(r), n_heads,
            static_cast<unsigned long long>(rows), hpc);
    return HQ_ERR_CUDA;
  }
  return HQ_OK;
}

static int alloc_weight(hq_ctx* ctx, Weight* w, int N, int K) {
  w->N = N;
  w->K = K;
  int rc = dev_alloc(ctx, &w->ptr, static_cast<size_t>(N) * K * ctx->wsize);
  if (rc) return rc;
  if (ctx->half) {
    if ((rc = make_map(ctx, &w->map, w->ptr, N, K, 64))) return rc;
    return make_pair_maps(ctx, &w->mapp, w->ptr, N, K);
  }
  return HQ_OK;
}
static int alloc_abuf(hq_ctx* ctx, ABuf* a, int rows, int K) {
  a->rows = (rows + 127) / 128 * 128;
  a->K = K;
  int rc = dev_alloc(ctx, &a->ptr, static_cast<size_t>(a->rows) * K * ctx->wsize);
  if (rc) return rc;
  if (ctx->half) {
    if ((rc = make_map(ctx, &a->map, a->ptr, a->rows, K, 128))) return rc;
    a->have3 = K >= 128;
    if (a->have3) return make_map3(ctx, &a->map3, a->ptr, a->rows, K, 128, 2);
  }
  return HQ_OK;
}
static int alloc_f32(hq_ctx* ctx, float** p, size_t n) { return dev_alloc(ctx, reinterpret_cast<void**>(p), n * 4); }

static void reg(hq_ctx* ctx, const std::string& name, void* dst, int is_weight, std::vector<int64_t> shape,
                bool ignored = false) {
  ParamSlot s;
  s.dst = dst;
  s.dst_is_weight = is_weight;
  s.shape = shape;
  s.ignored = ignored;
  ctx->params[name] = s;
}

static int build_block(hq_ctx* ctx, BlockW* b, const std::string& prefix) {
  const int D = ctx->D;
  int rc;
  if ((rc = alloc_weight(ctx, &b->qkv, 3 * D, D))) return rc;
  if ((rc = alloc_weight(ctx, &b->proj, D, D))) return rc;
  if ((rc = alloc_weight(ctx, &b->fc1, 4 * D, D))) return rc;
  if ((rc = alloc_weight(ctx, &b->fc2, D, 4 * D))) return rc;
  if ((rc = alloc_f32(ctx, &b->bqkv, 3 * D))) return rc;
  if ((rc = alloc_f32(ctx, &b->bproj, D))) return rc;
  if ((rc = alloc_f32(ctx, &b->b1, 4 * D))) return rc;
  if ((rc = alloc_f32(ctx, &b->b2, D))) return rc;
  float** lns[4] = {&b->ln1g, &b->ln1b, &b->ln2g, &b->ln2b};
  for (auto p : lns)
    if ((rc = alloc_f32(ctx, p, D))) return rc;
  const size_t wsz = ctx->wsize;
  char* wq = static_cast<char*>(b->qkv.ptr);
  // fused [q; k; v] rows (layers.py:43-50 keeps three separate nn.Linear modules)
  reg(ctx, prefix + ".attn.query.weight", wq, 1, {D, D});
  reg(ctx, prefix + ".attn.key.weight", wq + static_cast<size_t>(D) * D * wsz, 1, {D, D});
  reg(ctx, prefix + ".attn.value.weight", wq + static_cast<size_t>(2) * D * D * wsz, 1, {D, D});
  reg(ctx, prefix + ".attn.query.bias", b->bqkv, 0, {D});
  reg(ctx, prefix + ".attn.key.bias", b->bqkv + D, 0, {D});
  reg(ctx, prefix + ".attn.value.bias", b->bqkv + 2 * D, 0, {D});
  reg(ctx, prefix + ".attn.proj.weight", b->proj.ptr, 1, {D, D});
  reg(ctx, prefix + ".attn.proj.bias", b->bproj, 0, {D});
  reg(ctx, prefix + ".mlp.0.weight", b->fc1.ptr, 1, {4 * D, D});
  reg(ctx, prefix + ".mlp.0.bias", b->b1, 0, {4 * D});
  reg(ctx, prefix + ".mlp.2.weight", b->fc2.ptr, 1, {D, 4 * D});
  reg(ctx, prefix + ".mlp.2.bias", b->b2, 0, {D});
  reg(ctx, prefix + ".ln1.weight", b->ln1g, 0, {D});
  reg(ctx, prefix + ".ln1.bias", b->ln1b, 0, {D});
  reg(ctx, prefix + ".ln2.weight", b->ln2g, 0, {D});
  reg(ctx, prefix + ".ln2.bias", b->ln2b, 0, {D});
  return HQ_OK;
}

template <typename K>
static int set_smem(hq_ctx* ctx, K kernel, int bytes) {
  HQ_CUDA(ctx, cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
  return HQ_OK;
}

template <typename AT>
static int set_gemm_attrs(hq_ctx* ctx) {
  int rc;
#define HQ_SET(BN, EPI) \
  if ((rc = set_smem(ctx, gemm_tc_kernel<BN, EPI, AT, 1>, TcCfg<BN, 1>::SMEM_BYTES))) return rc; \
  if ((rc = set_smem(ctx, gemm_tc_kernel<BN, EPI, AT, 2>, TcCfg<BN, 2>::SMEM_BYTES))) return rc;
  HQ_SET(64, EPI_QKV) HQ_SET(64, EPI_RESID) HQ_SET(64, EPI_GELU) HQ_SET(64, EPI_F32) HQ_SET(64, EPI_SAMPLE)
  HQ_SET(128, EPI_QKV) HQ_SET(128, EPI_RESID) HQ_SET(128, EPI_GELU) HQ_SET(128, EPI_F32) HQ_SET(128, EPI_SAMPLE)
#undef HQ_SET
#define HQ_SET2(BN, EPI) \
  if ((rc = set_smem(ctx, gemm_tc2_kernel<BN, EPI, AT, 1>, Tc2Cfg<BN, 1>::SMEM_BYTES))) return rc; \
  if ((rc = set_smem(ctx, gemm_tc2_kernel<BN, EPI, AT, 2>, Tc2Cfg<BN, 2>::SMEM_BYTES))) return rc;
#define HQ_SET2_ALL(BN) HQ_SET2(BN, EPI_QKV) HQ_SET2(BN, EPI_RESID) HQ_SET2(BN, EPI_GELU) HQ_SET2(BN, EPI_F32) HQ_SET2(BN, EPI_SAMPLE)
  HQ_SET2_ALL(32) HQ_SET2_ALL(64) HQ_SET2_ALL(96) HQ_SET2_ALL(128) HQ_SET2_ALL(192) HQ_SET2_ALL(256)
#undef HQ_SET2_ALL
#undef HQ_SET2
  return HQ_OK;
}
static int set_gemm_attrs_for(hq_ctx* ctx) {
  return ctx->prec == HQ_PREC_F16 ? set_gemm_attrs<f16>(ctx) : set_gemm_attrs<bf16>(ctx);
}

// Calls f(AT()) with the activation type of precision `prec`: bf16, f16 (HQ_PREC_F16) or float (HQ_PREC_FP32).
template <typename F>
static void with_act(int prec, F&& f) {
  if (prec == HQ_PREC_BF16) f(bf16());
  else if (prec == HQ_PREC_F16) f(f16());
  else f(float());
}

static int get_encode_fn(hq_ctx* ctx, PFN_encodeTiled* fn) {
  void* p = nullptr;
  cudaDriverEntryPointQueryResult qres;
  HQ_CUDA(ctx, cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres));
  if (p == nullptr || qres != cudaDriverEntryPointSuccess) {
    set_err(ctx, "cuTensorMapEncodeTiled not available from the driver");
    return HQ_ERR_CUDA;
  }
  *fn = reinterpret_cast<PFN_encodeTiled>(p);
  return HQ_OK;
}

static int check_device(hq_ctx* ctx, int device) {
  int n = 0;
  HQ_CUDA(ctx, cudaGetDeviceCount(&n));
  if (device < 0 || device >= n) {
    set_err(ctx, "device %d out of range (%d visible)", device, n);
    return HQ_ERR_INVALID;
  }
  cudaDeviceProp prop;
  HQ_CUDA(ctx, cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10) {
    set_err(ctx, "libhqgraft is built for sm_100a only; device %d is sm_%d%d (no fallback path)", device, prop.major,
            prop.minor);
    return HQ_ERR_UNSUPPORTED;
  }
  return HQ_OK;
}

static void free_activations(hq_ctx* ctx);
static int reserve_impl(hq_ctx* ctx, int max_batch);

static int set_attn_attrs(hq_ctx* ctx) {
  int rc;
  if ((rc = set_smem(ctx, attention_decode_kernel<bf16>, 64 * 1024))) return rc;
  if ((rc = set_smem(ctx, attention_decode_kernel<f16>, 64 * 1024))) return rc;
  if ((rc = set_smem(ctx, attention_decode_kernel<float>, 64 * 1024))) return rc;
  if ((rc = set_smem(ctx, attention_decode_mma_kernel<bf16>, 112 * 1024))) return rc;
  return set_smem(ctx, attention_decode_mma_kernel<f16>, 112 * 1024);
}

// Head groups per image of the decode attention kernels: (image, group) work items, nh / groups heads (warps) each.
static int attn_groups(const hq_ctx* ctx, int nh) {
  int g = 0;
  for (int cand : {4, 3, 2, 1})
    if (nh % cand == 0 && nh / cand <= ATTD_MAXHPC) { g = cand; break; }
  // three heads per item where the head count allows it (24 heads: 8 groups, 2048 items at B = 256): the finer items balance
  // the tail of the launch better - 13.4 -> 12.8 us at 32 keys, +0.4-1.0 % end to end; 2, 4 or 12 heads per item measured
  // slower (profiles/r2_attn_groups_sweep.txt)
  if (nh % 3 == 0 && nh >= 12) g = nh / 3;
  const int v = ctx->dbg.attn_groups;                       // experiments: pin the number of head groups per image
  if (v >= 1 && nh % v == 0 && nh / v <= ATTD_MAXHPC) g = v;
  return g;
}

extern "C" int hq_abi_version(void) { return HQ_ABI_VERSION; }

extern "C" const char* hq_last_error(const hq_ctx* ctx) { return ctx ? ctx->err.c_str() : g_last_error.c_str(); }

extern "C" int hq_destroy(hq_ctx* ctx) {
  if (!ctx) return HQ_OK;
  cudaSetDevice(ctx->device);
  cudaDeviceSynchronize();
  free_activations(ctx);
  for (void* p : ctx->allocs) cudaFree(p);
  if (ctx->own_stream) cudaStreamDestroy(ctx->own_stream);
  delete ctx;
  return HQ_OK;
}

static void free_prefix_ws(hq_ctx* ctx) {
  for (void* p : ctx->pre_allocs) cudaFree(p);
  ctx->pre_allocs.clear();
  ctx->pre_bytes = 0;
  ctx->pre_rows = 0;
  ctx->pre_h = ABuf(); ctx->pre_att = ABuf(); ctx->pre_mlp = ABuf();
  ctx->pre_q = nullptr; ctx->pre_x = nullptr;
}

static void free_activations(hq_ctx* ctx) {
  for (auto& kv : ctx->graphs) cudaGraphExecDestroy(kv.second.exec);
  ctx->graphs.clear();
  free_prefix_ws(ctx);
  for (void* p : ctx->act_allocs) cudaFree(p);
  ctx->act_allocs.clear();
  ctx->act_bytes = 0;
  ctx->d_maps = nullptr;          // (an activation allocation) the op tables point into the freed buffers
  ctx->chain_index.clear();
  ctx->ops_used = 0;
}

// batch-sized state: activations, KV cache [L][B][Tc][D] x2, depth KV [Ld][B][5][D] x2, code buffers
static int reserve_alloc(hq_ctx* ctx, int max_batch);

// On failure (e.g. out of memory while growing the batch) the ctx keeps NO batch state: every batch-sized buffer is
// freed, the pointers are nulled and max_batch is 0, so validate_run rejects any run until a reserve succeeds.
static int reserve_impl(hq_ctx* ctx, int max_batch) {
  const int rc = reserve_alloc(ctx, max_batch);
  if (rc != HQ_OK) {
    const std::string why = ctx->err;
    cudaGetLastError();                        // clear the sticky-free allocation error
    free_activations(ctx);
    ctx->max_batch = 0;
    ctx->ws_rows = 0;
    ctx->kv_maps = false;
    ctx->h = ABuf(); ctx->att = ABuf(); ctx->mlp = ABuf();
    ctx->q = nullptr; ctx->x = nullptr; ctx->yd = nullptr; ctx->logits = nullptr; ctx->samp_part = nullptr; ctx->splitk_ws = nullptr;
    ctx->kc = ctx->vc = ctx->kd = ctx->vd = nullptr;
    ctx->cond = ctx->codes_top = ctx->codes_bot = ctx->codes_mid = nullptr;
    ctx->sos_override = nullptr;
    ctx->d_sp = nullptr;
    set_err(ctx, "hq_reserve_batch(%d) failed, the ctx holds no batch state until a reserve succeeds: %s", max_batch,
            why.c_str());
  }
  return rc;
}

static int reserve_alloc(hq_ctx* ctx, int max_batch) {
  int rc;
  if (max_batch < 1) {
    set_err(ctx, "max_batch must be >= 1");
    return HQ_ERR_INVALID;
  }
  HQ_CUDA(ctx, cudaSetDevice(ctx->device));
  HQ_CUDA(ctx, cudaDeviceSynchronize());
  free_activations(ctx);
  ctx->max_batch = max_batch;
  ctx->alloc_act = true;
  struct Guard { hq_ctx* c; ~Guard() { c->alloc_act = false; } } guard{ctx};
  const int D = ctx->D;
  const int B = max_batch;
  const int Mx = B * ctx->T0;                       // rows of the spatial residual stream (prefill for text)
  const int Mmax = (ctx->depth_rows * B > Mx) ? ctx->depth_rows * B : Mx;
  if ((rc = alloc_abuf(ctx, &ctx->h, Mmax, D))) return rc;
  if ((rc = alloc_abuf(ctx, &ctx->att, Mmax, D))) return rc;
  if ((rc = alloc_abuf(ctx, &ctx->mlp, Mmax, 4 * D))) return rc;
  if ((rc = dev_alloc(ctx, &ctx->q, static_cast<size_t>(Mmax) * D * ctx->wsize))) return rc;
  if ((rc = alloc_f32(ctx, &ctx->x, static_cast<size_t>(Mx) * D))) return rc;
  if ((rc = alloc_f32(ctx, &ctx->yd, static_cast<size_t>(ctx->depth_rows) * B * D))) return rc;
  if ((rc = alloc_f32(ctx, &ctx->logits, static_cast<size_t>(ctx->depth_rows < 4 ? 4 : ctx->depth_rows) * B * ctx->Vmax))) return rc;
  {
    float* sp2 = nullptr;
    if ((rc = alloc_f32(ctx, &sp2, static_cast<size_t>(ctx->depth_rows < 4 ? 4 : ctx->depth_rows) * B * ((ctx->Vmax + 31) / 32) * 2))) return rc;
    ctx->samp_part = reinterpret_cast<float2*>(sp2);
  }
  ctx->ws_rows = Mmax;
  if (ctx->half && (rc = alloc_f32(ctx, &ctx->splitk_ws, static_cast<size_t>(LN_MAXFOLD) * Mmax * D))) return rc;
  const size_t kvn = static_cast<size_t>(ctx->L) * B * ctx->Tc * D * ctx->wsize;
  if ((rc = dev_alloc(ctx, &ctx->kc, kvn))) return rc;
  if ((rc = dev_alloc(ctx, &ctx->vc, kvn))) return rc;
  ctx->kv_maps = false;
  if (ctx->half) {
    const int groups = attn_groups(ctx, ctx->nh);
    if (groups > 0) {
      const uint64_t rows = static_cast<uint64_t>(ctx->L) * B * ctx->Tc;
      if ((rc = make_kv_map(ctx, &ctx->kmap, ctx->kc, ctx->nh, rows, ctx->nh / groups))) return rc;
      if ((rc = make_kv_map(ctx, &ctx->vmap, ctx->vc, ctx->nh, rows, ctx->nh / groups))) return rc;
      ctx->kv_maps = true;
    }
  }
  const size_t kdn = static_cast<size_t>(ctx->Ld) * B * ctx->n_stack * D * ctx->wsize;
  if ((rc = dev_alloc(ctx, &ctx->kd, kdn))) return rc;
  if ((rc = dev_alloc(ctx, &ctx->vd, kdn))) return rc;
  if ((rc = dev_alloc(ctx, reinterpret_cast<void**>(&ctx->cond), static_cast<size_t>(B) * ctx->T0 * 8))) return rc;
  if ((rc = dev_alloc(ctx, reinterpret_cast<void**>(&ctx->codes_top), static_cast<size_t>(B) * ctx->Smax * 8))) return rc;
  if ((rc = dev_alloc(ctx, reinterpret_cast<void**>(&ctx->codes_bot),
                      static_cast<size_t>(B) * ctx->Smax * 8 * (ctx->levels == 3 ? 16 : 4)))) return rc;
  if (ctx->levels == 3 &&
      (rc = dev_alloc(ctx, reinterpret_cast<void**>(&ctx->codes_mid), static_cast<size_t>(B) * ctx->Smax * 32))) return rc;
  if ((rc = alloc_f32(ctx, &ctx->sos_override, static_cast<size_t>(Mx) * D))) return rc;
  if ((rc = dev_alloc(ctx, reinterpret_cast<void**>(&ctx->d_sp), sizeof(hq_sampling_params)))) return rc;
  if (ctx->prec == HQ_PREC_BF16) {
    // tensor-map table of the chain kernel (bf16 only): the three A buffers, then the six pair-tile maps of every GEMM weight
    std::vector<CUtensorMap> table;
    ABuf* abufs[3] = {&ctx->h, &ctx->att, &ctx->mlp};
    for (ABuf* a : abufs) {
      a->map_idx = static_cast<int>(table.size());
      table.push_back(a->map);
    }
    auto add_w = [&](Weight& w) {
      w.map_idx = static_cast<int>(table.size());
      for (int i = 0; i < 6; ++i) table.push_back(w.mapp.m[i]);
    };
    for (auto& b : ctx->blocks) { add_w(b.qkv); add_w(b.proj); add_w(b.fc1); add_w(b.fc2); }
    for (auto& b : ctx->depths) { add_w(b.qkv); add_w(b.proj); add_w(b.fc1); add_w(b.fc2); }
    add_w(ctx->head_top);
    add_w(ctx->head_bot);
    if (ctx->levels == 3) add_w(ctx->head_mid);
    if ((rc = dev_alloc(ctx, reinterpret_cast<void**>(&ctx->d_maps), table.size() * sizeof(CUtensorMap)))) return rc;
    HQ_CUDA(ctx, cudaMemcpy(ctx->d_maps, table.data(), table.size() * sizeof(CUtensorMap), cudaMemcpyHostToDevice));
  }
  return HQ_OK;
}

static int create_impl(hq_ctx* ctx, const hq_config* cfg, int device, int max_batch) {
  int rc;
  if (cfg->precision == HQ_PREC_TF32) {
    set_err(ctx, "HQ_PREC_TF32 is a stage-1 decoder precision (hq_s1_config); the sampler runs in bf16, fp16 or fp32");
    return HQ_ERR_INVALID;
  }
  if ((rc = check_device(ctx, device))) return rc;
  HQ_CUDA(ctx, cudaSetDevice(device));
  ctx->cfg = *cfg;
  ctx->device = device;
  ctx->max_batch = max_batch;
  ctx->prec = cfg->precision;
  ctx->half = cfg->precision != HQ_PREC_FP32;
  ctx->use_pdl = cfg->use_pdl != 0;
  ctx->wsize = ctx->half ? 2 : 4;
  const int D = ctx->D = cfg->embed_dim;
  ctx->nh = cfg->n_heads;
  ctx->L = cfg->n_layers;
  ctx->Ld = cfg->n_layers_depth;
  ctx->Vt = cfg->vocab_top;
  ctx->Vb = cfg->vocab_bot;
  ctx->Vmax = ctx->Vt > ctx->Vb ? ctx->Vt : ctx->Vb;
  ctx->levels = cfg->code_levels == 3 ? 3 : 2;
  if (cfg->code_levels != 0 && cfg->code_levels != 2 && cfg->code_levels != 3) {
    set_err(ctx, "code_levels must be 2 or 3 (got %d)", cfg->code_levels);
    return HQ_ERR_INVALID;
  }
  if (ctx->levels == 3) {
    ctx->Vm = cfg->vocab_mid;
    ctx->n_stack = 21;
    if (ctx->Vm > ctx->Vmax) ctx->Vmax = ctx->Vm;
    if (ctx->Vm < 64 || ctx->Vm % 64 != 0 || cfg->cond_kind == HQ_COND_TXT || cfg->model_type != HQ_MODEL_PARALLEL ||
        cfg->embedding_kind != HQ_EMB_TRANSFORMER1 || cfg->position_kind != HQ_POS_1D) {
      set_err(ctx, "code_levels == 3: the 'parallel-add' HQTransformer with class / unconditional sos, 'transformer1' embedding and "
                   "1-D positions is implemented (vocab_mid a multiple of 64)");
      return HQ_ERR_UNSUPPORTED;
    }
  }
  ctx->Smax = cfg->max_seq_len;
  const bool txt = cfg->cond_kind == HQ_COND_TXT;
  ctx->T0 = txt ? cfg->ctx_len_txt : 1;
  ctx->Tc = ctx->T0 + ctx->Smax - 1;
  if (max_batch < 1 || D < 64 || D % 64 != 0 || ctx->nh * 64 != D) {
    set_err(ctx, "unsupported shape: embed_dim=%d n_heads=%d (head size must be 64), max_batch=%d", D, ctx->nh, max_batch);
    return HQ_ERR_UNSUPPORTED;
  }
  if (ctx->Vt % 64 != 0 || ctx->Vb % 64 != 0 || ctx->Vmax > 32768) {
    set_err(ctx, "unsupported vocabulary sizes %d / %d (multiples of 64, <= 32768)", ctx->Vt, ctx->Vb);
    return HQ_ERR_UNSUPPORTED;
  }
  if (ctx->Tc > ATT_MAX_KEYS || ctx->Smax < 1 || ctx->Smax > cfg->ctx_len_img) {
    set_err(ctx, "unsupported lengths: max_seq_len=%d ctx_len_img=%d ctx_len_txt=%d (cache length %d > %d)", ctx->Smax,
            cfg->ctx_len_img, cfg->ctx_len_txt, ctx->Tc, ATT_MAX_KEYS);
    return HQ_ERR_UNSUPPORTED;
  }
  if (cfg->cond_kind < 0 || cfg->cond_kind > 2 || cfg->precision < HQ_PREC_BF16 || cfg->precision > HQ_PREC_F16) {
    set_err(ctx, "bad cond_kind / precision");
    return HQ_ERR_INVALID;
  }
  if (cfg->model_type < 0 || cfg->model_type > 2 || cfg->embedding_kind < 0 || cfg->embedding_kind > 1 ||
      cfg->position_kind < 0 || cfg->position_kind > 1) {
    set_err(ctx, "bad model_type / embedding_kind / position_kind");
    return HQ_ERR_INVALID;
  }
  if (cfg->embedding_kind == HQ_EMB_REDUCE && D % 16 != 0) {
    set_err(ctx, "embedding_type 'reduce' needs embed_dim %% 16 == 0 (four D/4-wide bottom embeddings)");
    return HQ_ERR_UNSUPPORTED;
  }
  ctx->depth_rows = ctx->levels == 3 ? 16 : (cfg->model_type == HQ_MODEL_BIDIRECTIONAL ? 5 : 4);
  if (cfg->position_kind == HQ_POS_2D) {
    int H = 1;
    while ((H + 1) * (H + 1) <= cfg->ctx_len_img) ++H;        // int(math.sqrt(ctx_len_img)), hierarchical_ar.py:122
    ctx->Hpos = H;
  }
  if (ctx->half) {
    if ((rc = get_encode_fn(ctx, &ctx->encode))) return rc;
    if ((rc = set_gemm_attrs_for(ctx))) return rc;
  }
  if ((rc = set_attn_attrs(ctx))) return rc;
  if ((rc = dev_alloc(ctx, reinterpret_cast<void**>(&ctx->att_sched), 16))) return rc;
  HQ_CUDA(ctx, cudaMemset(ctx->att_sched, 0, 16));
  HQ_CUDA(ctx, cudaDeviceGetAttribute(&ctx->num_sms, cudaDevAttrMultiProcessorCount, device));
  HQ_CUDA(ctx, cudaStreamCreateWithFlags(&ctx->own_stream, cudaStreamNonBlocking));
  if (ctx->prec == HQ_PREC_BF16 && cfg->use_chain && !ctx->dbg.no_chain) {
    // persistent chain kernel (bf16 engine only; the fp16 and fp32 engines ignore use_chain): every launch uses the same
    // grid of co-resident CTA pairs (its ops are separated by a grid barrier, so a CTA that is not resident would deadlock
    // the rest)
    if ((rc = set_smem(ctx, chain_kernel, CH_SMEM_BYTES))) return rc;
    cudaLaunchConfig_t lc;
    memset(&lc, 0, sizeof(lc));
    lc.gridDim = dim3(2 * 74);
    lc.blockDim = dim3(CH_THREADS);
    lc.dynamicSmemBytes = CH_SMEM_BYTES;
    int clusters = 0;
    HQ_CUDA(ctx, cudaOccupancyMaxActiveClusters(&clusters, chain_kernel, &lc));
    if (clusters > ctx->num_sms / 2) clusters = ctx->num_sms / 2;
    if (clusters >= 32) {
      ctx->chain_grid = 2 * clusters;
      ctx->ops_cap = 2048;
      if ((rc = dev_alloc(ctx, reinterpret_cast<void**>(&ctx->d_ops), sizeof(ChainOp) * ctx->ops_cap))) return rc;
      if ((rc = dev_alloc(ctx, reinterpret_cast<void**>(&ctx->d_chain_bar), 256))) return rc;
      ctx->chain_ok = true;
    }
  }

  // ---- parameters ----
  ctx->blocks.resize(ctx->L);
  ctx->depths.resize(ctx->Ld);
  for (int i = 0; i < ctx->L; ++i)
    if ((rc = build_block(ctx, &ctx->blocks[i], "blocks." + std::to_string(i)))) return rc;
  for (int i = 0; i < ctx->Ld; ++i)
    if ((rc = build_block(ctx, &ctx->depths[i], "depths." + std::to_string(i)))) return rc;
  if ((rc = alloc_weight(ctx, &ctx->head_top, ctx->Vt, D))) return rc;
  if ((rc = alloc_weight(ctx, &ctx->head_bot, ctx->Vb, D))) return rc;
  struct F32P { const char* name; float** p; std::vector<int64_t> shape; };
  std::vector<F32P> f32s;
  if (ctx->levels == 3) {
    // ---- HQTransformer state_dict (hqtransformer.py:24-166), decoding_type 'parallel-add' ----
    if ((rc = alloc_weight(ctx, &ctx->head_mid, ctx->Vm, D))) return rc;
    reg(ctx, "head_levels.0.weight", ctx->head_top.ptr, 1, {ctx->Vt, D});
    reg(ctx, "head_levels.1.weight", ctx->head_mid.ptr, 1, {ctx->Vm, D});
    reg(ctx, "head_levels.2.weight", ctx->head_bot.ptr, 1, {ctx->Vb, D});
    f32s = {
        {"sos_depth", &ctx->sos_depth, {1, 1, D}},
        {"tok_emb_levels.0.weight", &ctx->E_top, {ctx->Vt, D}},
        {"tok_emb_levels.1.weight", &ctx->E_mid, {ctx->Vm, D}},
        {"tok_emb_levels.2.weight", &ctx->E_bot, {ctx->Vb, D}},
        {"pos_emb_emb.weight", &ctx->P_emb, {21, D}},
        {"pos_emb_top.weight", &ctx->P_top, {cfg->ctx_len_img, D}},
        {"tok_emb_depth_levels.0.weight", &ctx->E_top_depth, {ctx->Vt, D}},
        {"tok_emb_depth_levels.1.weight", &ctx->E_mid_depth, {ctx->Vm, D}},
        {"pos_emb_depths.0.weight", &ctx->P_depth, {4, D}},
        {"pos_emb_depths.1.weight", &ctx->P_depth2, {16, D}},
        {"ln_f.weight", &ctx->lnf_g, {D}}, {"ln_f.bias", &ctx->lnf_b, {D}},
        {"ln_levels.0.weight", &ctx->lnt_g, {D}}, {"ln_levels.0.bias", &ctx->lnt_b, {D}},
        {"ln_levels.1.weight", &ctx->lnm_g, {D}}, {"ln_levels.1.bias", &ctx->lnm_b, {D}},
        {"ln_levels.2.weight", &ctx->lnb_g, {D}}, {"ln_levels.2.bias", &ctx->lnb_b, {D}},
    };
    // the bottom level's depth embedding exists in the state_dict and is never read when sampling (:521-524)
    reg(ctx, "tok_emb_depth_levels.2.weight", nullptr, 0, {ctx->Vb, D}, true);
  } else {
    reg(ctx, "head_top.weight", ctx->head_top.ptr, 1, {ctx->Vt, D});
    reg(ctx, "head_bot.weight", ctx->head_bot.ptr, 1, {ctx->Vb, D});
    f32s = {
        {"sos_depth", &ctx->sos_depth, {1, 1, D}},
        {"tok_emb_top.weight", &ctx->E_top, {ctx->Vt, D}},
        {"tok_emb_top_depth.weight", &ctx->E_top_depth, {ctx->Vt, D}},
        {"pos_emb_depth.weight", &ctx->P_depth, {5, D}},
        {"ln_f.weight", &ctx->lnf_g, {D}}, {"ln_f.bias", &ctx->lnf_b, {D}},
        {"ln_top.weight", &ctx->lnt_g, {D}}, {"ln_top.bias", &ctx->lnt_b, {D}},
        {"ln_bot.weight", &ctx->lnb_g, {D}}, {"ln_bot.bias", &ctx->lnb_b, {D}},
    };
    if (cfg->embedding_kind == HQ_EMB_REDUCE) {               // hierarchical_ar.py:85-88
      f32s.push_back({"tok_emb_bot.weight", &ctx->E_bot, {ctx->Vb, D / 4}});
    } else {                                                   // :97-103
      f32s.push_back({"tok_emb_bot.weight", &ctx->E_bot, {ctx->Vb, D}});
      f32s.push_back({"pos_emb_emb.weight", &ctx->P_emb, {5, D}});
    }
    if (cfg->position_kind == HQ_POS_2D) {                     // :121-125
      f32s.push_back({"pos_emb_top_h.weight", &ctx->P_top_h, {ctx->Hpos, D}});
      f32s.push_back({"pos_emb_top_w.weight", &ctx->P_top_w, {ctx->Hpos, D}});
    } else {
      f32s.push_back({"pos_emb_top.weight", &ctx->P_top, {cfg->ctx_len_img, D}});
    }
    if (cfg->model_type == HQ_MODEL_TOP2BOT) f32s.push_back({"tok_emb_bot_depth.weight", &ctx->E_bot_depth, {ctx->Vb, D}});
    // present in the reference state_dict, never read when sampling model_type='parallel' (SURVEY.md 8a a7)
    if (cfg->model_type != HQ_MODEL_TOP2BOT) reg(ctx, "tok_emb_bot_depth.weight", nullptr, 0, {ctx->Vb, D}, true);
  }
  if (cfg->cond_kind == HQ_COND_CLS) f32s.push_back({"sos.weight", &ctx->sos_table, {cfg->n_classes, D}});
  if (cfg->cond_kind == HQ_COND_UNCOND) f32s.push_back({"sos", &ctx->sos_table, {1, 1, D}});
  if (txt) {
    f32s.push_back({"tok_emb_txt.weight", &ctx->E_txt, {cfg->vocab_txt, D}});
    f32s.push_back({"pos_emb_txt.weight", &ctx->P_txt, {cfg->ctx_len_txt, D}});
  }
  for (auto& f : f32s) {
    size_t n = 1;
    for (auto s : f.shape) n *= static_cast<size_t>(s);
    if ((rc = alloc_f32(ctx, f.p, n))) return rc;
    reg(ctx, f.name, *f.p, 0, f.shape);
  }
  if (txt) {
    reg(ctx, "head_txt.weight", nullptr, 0, {cfg->vocab_txt, D}, true);
    reg(ctx, "ln_txt.weight", nullptr, 0, {D}, true);
    reg(ctx, "ln_txt.bias", nullptr, 0, {D}, true);
  }

  return reserve_impl(ctx, max_batch);
}

extern "C" int hq_create(const hq_config* cfg, int device, int max_batch, hq_ctx** out) {
  if (!cfg || !out) {
    set_err(nullptr, "hq_create: null argument");
    return HQ_ERR_INVALID;
  }
  *out = nullptr;
  hq_ctx* ctx = new hq_ctx();
  int rc = create_impl(ctx, cfg, device, max_batch);
  if (rc != HQ_OK) {
    g_last_error = ctx->err;
    free_activations(ctx);
    for (void* p : ctx->allocs) cudaFree(p);
      if (ctx->own_stream) cudaStreamDestroy(ctx->own_stream);
    delete ctx;
    return rc;
  }
  *out = ctx;
  return HQ_OK;
}

// ------------------------------------------------------------------------------------------------
// parameter loading
// ------------------------------------------------------------------------------------------------
template <typename S, typename Dt>
__global__ void convert_kernel(const S* __restrict__ s, Dt* __restrict__ d, size_t n) {
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < n;
       i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    float v;
    if (sizeof(S) == 4) v = *reinterpret_cast<const float*>(&s[i]);
    else if (std::is_same<S, bf16>::value) v = __bfloat162float(*reinterpret_cast<const bf16*>(&s[i]));
    else v = __half2float(*reinterpret_cast<const __half*>(&s[i]));
    d[i] = ActT<Dt>::from_f(v);
  }
}

// dst_prec: the storage type of the destination (HQ_PREC_BF16 | HQ_PREC_F16 | HQ_PREC_FP32)
template <typename S>
static void launch_convert(const void* src, void* dst, int dst_prec, size_t n) {
  const int grid = static_cast<int>((n + 255) / 256 > 4096 ? 4096 : (n + 255) / 256);
  with_act(dst_prec, [&](auto tag) {
    using Dt = decltype(tag);
    convert_kernel<S, Dt><<<grid, 256>>>(static_cast<const S*>(src), static_cast<Dt*>(dst), n);
  });
}

extern "C" int hq_load_param(hq_ctx* ctx, const char* name, const void* data, int dtype, const int64_t* shape, int ndim,
                             int is_device) {
  if (!ctx || !name || !data || !shape) {
    set_err(ctx, "hq_load_param: null argument");
    return HQ_ERR_INVALID;
  }
  HQ_CUDA(ctx, cudaSetDevice(ctx->device));
  auto it = ctx->params.find(name);
  if (it == ctx->params.end()) {
    set_err(ctx, "unexpected key in state_dict: \"%s\"", name);
    return HQ_ERR_INVALID;
  }
  ParamSlot& s = it->second;
  bool ok = static_cast<size_t>(ndim) == s.shape.size();
  for (int i = 0; ok && i < ndim; ++i) ok = shape[i] == s.shape[i];
  if (!ok) {
    std::string want, got;
    for (auto v : s.shape) want += std::to_string(v) + ",";
    for (int i = 0; i < ndim; ++i) got += std::to_string(shape[i]) + ",";
    set_err(ctx, "size mismatch for %s: expected [%s] got [%s]", name, want.c_str(), got.c_str());
    return HQ_ERR_INVALID;
  }
  if (dtype < HQ_F32 || dtype > HQ_F16) {
    set_err(ctx, "bad dtype %d for %s", dtype, name);
    return HQ_ERR_INVALID;
  }
  s.loaded = true;
  if (s.ignored) return HQ_OK;
  size_t n = 1;
  for (auto v : s.shape) n *= static_cast<size_t>(v);
  const size_t esz = dtype == HQ_F32 ? 4 : 2;
  const void* src = data;
  void* staged = nullptr;
  if (!is_device) {
    HQ_CUDA(ctx, cudaMalloc(&staged, n * esz));
    cudaError_t e = cudaMemcpy(staged, data, n * esz, cudaMemcpyHostToDevice);
    if (e != cudaSuccess) {
      cudaFree(staged);
      set_err(ctx, "cudaMemcpy H2D failed for %s: %s", name, cudaGetErrorString(e));
      return HQ_ERR_CUDA;
    }
    src = staged;
  }
  const int dst_prec = s.dst_is_weight ? ctx->prec : HQ_PREC_FP32;
  if (dtype == HQ_F32) launch_convert<float>(src, s.dst, dst_prec, n);
  else if (dtype == HQ_BF16) launch_convert<bf16>(src, s.dst, dst_prec, n);
  else launch_convert<__half>(src, s.dst, dst_prec, n);
  cudaError_t e = cudaDeviceSynchronize();
  if (staged) cudaFree(staged);
  if (e != cudaSuccess) {
    set_err(ctx, "parameter conversion failed for %s: %s", name, cudaGetErrorString(e));
    return HQ_ERR_CUDA;
  }
  return HQ_OK;
}

extern "C" int hq_params_complete(hq_ctx* ctx) {
  if (!ctx) return HQ_ERR_INVALID;
  std::string missing;
  int n = 0;
  for (auto& kv : ctx->params)
    if (!kv.second.loaded && !kv.second.ignored) {
      if (n < 8) missing += (n ? ", " : "") + kv.first;
      ++n;
    }
  if (n) {
    set_err(ctx, "missing %d key(s) in state_dict: %s%s", n, missing.c_str(), n > 8 ? ", ..." : "");
    return HQ_ERR_STATE;
  }
  return HQ_OK;
}

extern "C" int hq_reserve_batch(hq_ctx* ctx, int max_batch) {
  if (!ctx) return HQ_ERR_INVALID;
  return reserve_impl(ctx, max_batch);
}
extern "C" int hq_max_batch(const hq_ctx* ctx) { return ctx ? ctx->max_batch : 0; }

extern "C" int64_t hq_last_launch_count(const hq_ctx* ctx) { return ctx ? ctx->last_launches : 0; }
extern "C" int64_t hq_chain_launch_count(const hq_ctx* ctx) { return ctx ? ctx->chain_launches : 0; }
extern "C" size_t hq_device_bytes(const hq_ctx* ctx) { return ctx ? ctx->device_bytes + ctx->act_bytes + ctx->pre_bytes : 0; }

// ------------------------------------------------------------------------------------------------
// launch helpers
// ------------------------------------------------------------------------------------------------


// ------------------------------------------------------------------------------------------------
// launch helper: every kernel of the loop goes through cudaLaunchKernelEx so that the programmatic-dependent-launch
// attribute can be attached (the kernels call griddepcontrol.launch_dependents / .wait themselves).
// ------------------------------------------------------------------------------------------------
template <typename... KArgs, typename... Args>
static void launch_k(hq_ctx* ctx, cudaStream_t st, const char* tag, void (*kernel)(int, KArgs...), dim3 grid, dim3 block,
                     size_t smem, Args&&... args) {
  if (ctx->chain_mode == hq_ctx::CHAIN_PLAN) {     // planning pass of the chain kernel: op tables only
    ctx->tag_suffix.clear();
    return;
  }
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = (ctx->use_pdl && !ctx->full_dependency_next) ? 1 : 0;
  ctx->full_dependency_next = false;
  // experiments only: HQ_ABLATE=tag[,tag...] drops every launch whose tag starts with one of the names, to read a
  // kernel family's MARGINAL cost in the PDL-overlapped loop off the step time (results are garbage, timing is not)
  const char* ablate = ctx->dbg.ablate.empty() ? nullptr : ctx->dbg.ablate.c_str();
  if (ablate != nullptr) {
    const size_t n = strlen(tag);
    for (const char* p = ablate; *p;) {
      const char* e = strchr(p, ',');
      const size_t len = e ? static_cast<size_t>(e - p) : strlen(p);
      if (len > 0 && len <= n && strncmp(p, tag, len) == 0) {
        ctx->tag_suffix.clear();
        return;
      }
      p += len + (e ? 1 : 0);
    }
  }
  int trace_id = -1;
  if (ctx->tracing && static_cast<int>(ctx->trace_tags.size()) < ctx->trace_cap) {
    trace_id = static_cast<int>(ctx->trace_tags.size());
    ctx->trace_tags.push_back(std::string(tag) + ctx->tag_suffix);
  }
  ctx->tag_suffix.clear();
  cudaError_t e = cudaLaunchKernelEx(&cfg, kernel, trace_id, static_cast<KArgs>(args)...);
  ++ctx->launches;
  if (e == cudaSuccess) e = cudaGetLastError();
  if (e != cudaSuccess && ctx->launch_err == cudaSuccess) ctx->launch_err = e;
}

// ------------------------------------------------------------------------------------------------
// persistent chain kernel: op recording and launch (chain.cuh)
// ------------------------------------------------------------------------------------------------
static bool chain_enabled(const hq_ctx* ctx, int B) {
  const int min_b = ctx->dbg.chain_min_batch > 0 ? ctx->dbg.chain_min_batch : 129;   // every GEMM on CTA-pair tiles
  return ctx->chain_ok && ctx->levels == 2 && ctx->cfg.model_type == HQ_MODEL_PARALLEL && ctx->d_maps != nullptr && B >= min_b && ctx->D <= LN_MAXV * LN_THREADS * 4 &&
         ctx->chain_mode != hq_ctx::CHAIN_OFF;
}

static ChainOp* chain_push(hq_ctx* ctx, int kind, const std::string& tag) {
  ChainOp op;
  memset(&op, 0, sizeof(op));
  op.kind = kind;
  ctx->rec.push_back(op);
  ctx->rec_tags.push_back(tag);
  return &ctx->rec.back();
}

static void chain_begin(hq_ctx* ctx, int t0, int pos, int S) {
  ctx->recording = true;
  ctx->rec.clear();
  ctx->rec_tags.clear();
  ctx->chain_rt.t0 = t0;
  ctx->chain_rt.pos = pos;
  ctx->chain_rt.S = S;
}

// Launches the ops recorded so far as ONE chain_kernel launch (recording stays on: the caller may go on appending).
// PLAN pass: the op table is deduplicated by content and uploaded; RUN pass: it must already be on the device.
static void chain_flush(hq_ctx* ctx, cudaStream_t st) {
  const int n = static_cast<int>(ctx->rec.size());
  if (n == 0) return;
  const std::string key(reinterpret_cast<const char*>(ctx->rec.data()), sizeof(ChainOp) * static_cast<size_t>(n));
  auto it = ctx->chain_index.find(key);
  if (ctx->chain_mode == hq_ctx::CHAIN_PLAN) {
    if (it == ctx->chain_index.end()) {
      if (ctx->ops_used + n > ctx->ops_cap) {
        if (ctx->launch_err == cudaSuccess) ctx->launch_err = cudaErrorMemoryAllocation;
      } else {
        cudaError_t e = cudaMemcpy(ctx->d_ops + ctx->ops_used, ctx->rec.data(), sizeof(ChainOp) * static_cast<size_t>(n),
                                   cudaMemcpyHostToDevice);
        if (e != cudaSuccess && ctx->launch_err == cudaSuccess) ctx->launch_err = e;
        ctx->chain_index.emplace(key, ctx->ops_used);
        ctx->ops_used += n;
      }
    }
  } else {
    if (it == ctx->chain_index.end()) {
      if (ctx->launch_err == cudaSuccess) ctx->launch_err = cudaErrorInvalidValue;   // not planned: a host logic error
    } else {
      ChainRt rt = ctx->chain_rt;
      rt.bar = ctx->d_chain_bar;
      rt.bar_base = ctx->chain_epoch;
      rt.trace_base = -1;
      rt.no_l2_prefetch = ctx->dbg.chain_no_l2pf;
      rt.phase_op = (ctx->phase_launch >= 0 && ctx->chain_launches_run == ctx->phase_launch) ? ctx->phase_op : -1;
      ++ctx->chain_launches_run;
      if (ctx->tracing && static_cast<int>(ctx->trace_tags.size()) + n <= ctx->trace_cap) {
        rt.trace_base = static_cast<int>(ctx->trace_tags.size());
        for (int i = 0; i < n; ++i) {
          ctx->trace_tags.push_back(ctx->rec_tags[i]);
          ctx->trace_chain_cont.resize(ctx->trace_tags.size(), 0);
          ctx->trace_chain_cont.back() = i > 0 ? 1 : 0;
        }
      }
      const bool was_tracing = ctx->tracing;
      ctx->tracing = false;                        // the launch itself takes no timeline entry: its ops do
      launch_k(ctx, st, "chain", chain_kernel, dim3(ctx->chain_grid), dim3(CH_THREADS), CH_SMEM_BYTES,
               static_cast<const ChainOp*>(ctx->d_ops + it->second), n, static_cast<const CUtensorMap*>(ctx->d_maps), rt);
      ctx->tracing = was_tracing;
      ctx->chain_epoch += static_cast<unsigned long long>(n) * static_cast<unsigned long long>(ctx->chain_grid);
      ++ctx->chain_launches;
      ctx->chain_ops += n;
    }
  }
  ctx->rec.clear();
  ctx->rec_tags.clear();
}

static void chain_end(hq_ctx* ctx, cudaStream_t st) {
  chain_flush(ctx, st);
  ctx->recording = false;
}

template <int EPI>
static const char* gemm_tag(int M) {
  (void)M;
  return EPI == EPI_QKV ? "gemm_qkv" : (EPI == EPI_RESID ? "gemm_resid" : (EPI == EPI_GELU ? "gemm_fc1_gelu" : "gemm_head"));
}

// Cost model behind the tile / split-K choices (cycles; constants fitted to profiles/r1_gemm_plan_sweep.txt, measured
// with ONE GEMM CTA per SM): a wave of <= 74 CTA pairs costs a fixed ~11k cycles (launch ramp, prologue, first TMA round
// trip, epilogue, teardown) plus, per 64-wide k-block, the larger of the operand ingest at ~42.6 B/clk/SM and the tensor
// pipe time; wide tiles pay for their extra epilogue chunks.
static double pair_gemm_cost(int M, int N, int K, int bn, int splits) {
  const int pairs = ((M + 255) / 256) * (N / bn) * splits;
  const double waves = static_cast<double>((pairs + 73) / 74);
  const double ingest = (16384.0 + 64.0 * bn) / 42.6, mma = 2.0 * bn;
  // split-K slices also write M x N fp32 partials each (L2 write bandwidth, ~40 B/clk/SM: the term that makes 2 slices
  // beat 3 for proj at 1024 rows, 8.3 vs 9.3 us, profiles/r2_splitk_final.txt)
  const double partials = splits > 1 ? static_cast<double>(M) * N * 4.0 * splits / 5920.0 : 0.0;
  return waves * ((K / 64 / splits) * (ingest > mma ? ingest : mma) + 11000.0) + (splits > 1 ? 400.0 * splits : 0.0) +
         partials + 16.0 * bn;
}

// Width of the CTA-pair tile (256 x BN) for an [M, N] output
static int pick_pair_bn(int M, int N, int K) {
  static const int cand[6] = {256, 192, 128, 96, 64, 32};
  int best = 0;
  double best_cost = 1e30;
  for (int bn : cand) {
    if (N % bn != 0) continue;
    const double cost = pair_gemm_cost(M, N, K, bn, 1);
    if (cost < best_cost) {
      best_cost = cost;
      best = bn;
    }
  }
  return best;
}

// The tcgen05 GEMM of the 2-byte engines (AT = bf16 | f16) on the operands' tensor maps.
template <int EPI, typename AT>
static void gemm_tc(hq_ctx* ctx, cudaStream_t st, const CUtensorMap& mA, const CUtensorMap* mA3, const CUtensorMap& mW64,
                    const PairMaps& mWp, int w_row_off, int M, int N, int K, const EpiParams<AT>& ep,
                    int splits = 1, int bn_hint = 0, int ia = -1, int iw = -1) {
  int bn = ctx->dbg.force_bn ? ctx->dbg.force_bn : bn_hint;
  if (bn == 0) bn = (M > 128) ? pick_pair_bn(M, N, K) : 0;
  if (bn_hint == 0 && !ctx->dbg.force_bn && ctx->dbg.bn_m256 > 0 && M > 128 && M <= 256 && N % ctx->dbg.bn_m256 == 0) bn = ctx->dbg.bn_m256;
  if (ctx->recording) {
    // an op of the persistent chain kernel (bf16): CTA-pair tiles only (chain_enabled guarantees M > 128)
    if (!std::is_same<AT, bf16>::value || bn <= 0 || N % bn != 0 || ia < 0 || iw < 0 || (K / 64) % splits != 0) {
      if (ctx->launch_err == cudaSuccess) ctx->launch_err = cudaErrorInvalidValue;
      return;
    }
    char buf[64];
    snprintf(buf, sizeof(buf), "%s:%dx%dx%d:s%d", ctx->gemm_tag_override ? ctx->gemm_tag_override : gemm_tag<EPI>(M), M, N, K,
             splits);
    ctx->gemm_tag_override = nullptr;
    ChainOp* op = chain_push(ctx, CH_OP_GEMM, buf);
    op->flags = ctx->rec_flags;
    op->map_a = ia;
    op->map_w = iw + PairMaps::index(bn);
    op->M = M; op->N = N; op->K = K; op->bn = bn; op->splits = splits; op->epi = EPI; op->w_row_off = w_row_off;
    if constexpr (std::is_same<AT, bf16>::value) op->ep = ep;   // the chain kernel is bf16 only (refused above otherwise)
    if (op->flags & CH_F_T0_RT) op->ep.t0 = 0;
    return;
  }
  if (ctx->tracing) {
    char buf[48];
    snprintf(buf, sizeof(buf), ":%dx%dx%d:s%d", M, N, K, splits);
    ctx->tag_suffix = buf;
  }
  const char* tag = ctx->gemm_tag_override ? ctx->gemm_tag_override : gemm_tag<EPI>(M);
  ctx->gemm_tag_override = nullptr;
  if (bn > 0 && N % bn == 0) {
    const int tiles = (N / bn) * ((M + 255) / 256) * splits;
    dim3 grid(2 * (tiles < 74 ? tiles : 74));               // persistent: at most one CTA pair per SM pair
    // two k-blocks per ring stage (3-D boxes) whenever every tile's K range holds an even number of k-blocks
    const bool ks2 = mA3 != nullptr && mWp.have3 && !ctx->dbg.gemm_ks1 && ((K / 64) / splits) % 2 == 0;
#define HQ_LAUNCH2(BN)                                                                                             \
  case BN:                                                                                                         \
    if (ks2)                                                                                                       \
      launch_k(ctx, st, tag, gemm_tc2_kernel<BN, EPI, AT, 2>, grid, dim3(Tc2Cfg<BN, 2>::THREADS), Tc2Cfg<BN, 2>::SMEM_BYTES, *mA3,  \
               mWp.m3[PairMaps::index(BN)], M, N, K, w_row_off, splits, ep);                                       \
    else                                                                                                           \
      launch_k(ctx, st, tag, gemm_tc2_kernel<BN, EPI, AT, 1>, grid, dim3(Tc2Cfg<BN, 1>::THREADS), Tc2Cfg<BN, 1>::SMEM_BYTES, mA,  \
               mWp.m[PairMaps::index(BN)], M, N, K, w_row_off, splits, ep);                                        \
    break;
    switch (bn) {
      HQ_LAUNCH2(32) HQ_LAUNCH2(64) HQ_LAUNCH2(96) HQ_LAUNCH2(128) HQ_LAUNCH2(192) HQ_LAUNCH2(256)
      default: ctx->launch_err = cudaErrorInvalidValue;
    }
#undef HQ_LAUNCH2
    return;
  }
  const int mt = (M + 127) / 128;
  const bool wide = bn == -128 || (bn != -64 && (N % 128 == 0) && (mt * (N / 128) >= 120));
  const int tbn = wide ? 128 : 64;
  // two k-blocks per ring stage: the W tile of tbn rows is the pair map of width 2 * tbn (box {64, tbn, 2})
  const bool ks2 = mA3 != nullptr && mWp.have3 && !ctx->dbg.gemm_ks1 && ((K / 64) / splits) % 2 == 0 && N >= 2 * tbn;
  dim3 grid(N / tbn, mt, splits);
  if (wide) {
    if (ks2)
      launch_k(ctx, st, tag, gemm_tc_kernel<128, EPI, AT, 2>, grid, dim3(192), TcCfg<128, 2>::SMEM_BYTES, *mA3,
               mWp.m3[PairMaps::index(256)], M, N, K, w_row_off, ep);
    else
      launch_k(ctx, st, tag, gemm_tc_kernel<128, EPI, AT, 1>, grid, dim3(192), TcCfg<128, 1>::SMEM_BYTES, mA, mW64, M, N, K,
               w_row_off, ep);
  } else {
    if (ks2)
      launch_k(ctx, st, tag, gemm_tc_kernel<64, EPI, AT, 2>, grid, dim3(192), TcCfg<64, 2>::SMEM_BYTES, *mA3,
               mWp.m3[PairMaps::index(128)], M, N, K, w_row_off, ep);
    else
      launch_k(ctx, st, tag, gemm_tc_kernel<64, EPI, AT, 1>, grid, dim3(192), TcCfg<64, 1>::SMEM_BYTES, mA, mW64, M, N, K,
               w_row_off, ep);
  }
}

template <int EPI>
static void gemm_f32(hq_ctx* ctx, cudaStream_t st, const float* A, const float* W, int M, int N, int K,
                     const EpiParams<float>& ep) {
  dim3 grid((N + 127) / 128, (M + 63) / 64);
  launch_k(ctx, st, gemm_tag<EPI>(M), gemm_simt_kernel<EPI>, grid, dim3(256), 0, A, W, M, N, K, ep);
}

template <int EPI, typename AT>
static void gemm_any(hq_ctx* ctx, cudaStream_t st, const ABuf& A, const Weight& W, int w_row_off, int M, int N, int K,
                     const EpiParams<AT>& ep) {
  gemm_tc<EPI, AT>(ctx, st, A.map, A.have3 ? &A.map3 : nullptr, W.map, W.mapp, w_row_off, M, N, K, ep, 1, 0, A.map_idx, W.map_idx);
}
template <int EPI>
static void gemm_any(hq_ctx* ctx, cudaStream_t st, const ABuf& A, const Weight& W, int w_row_off, int M, int N, int K,
                     const EpiParams<float>& ep) {
  gemm_f32<EPI>(ctx, st, static_cast<const float*>(A.ptr),
                static_cast<const float*>(W.ptr) + static_cast<size_t>(w_row_off) * K, M, N, K, ep);
}

// Pending split-K partial sums of the last RESID GEMM: the next LayerNorm on that residual stream folds them in.
struct Fold {
  const float* partial = nullptr;
  int n = 0;
  size_t stride = 0;
  const float* bias = nullptr;
};

template <typename AT>
static void layernorm_act(hq_ctx* ctx, cudaStream_t st, float* x, const float* g, const float* b, AT* out, int rows,
                          Fold* fold = nullptr) {
  Fold f = fold ? *fold : Fold();
  if (ctx->recording) {
    ChainOp* op = chain_push(ctx, CH_OP_LN, "layernorm");
    op->flags = sizeof(AT) == 4 ? CH_F_OUT_F32 : 0;
    op->x = x; op->gamma = g; op->beta = b; op->add = nullptr; op->out = out;
    op->rows = rows; op->in_mul = 1; op->in_off = 0; op->D = ctx->D;
    op->fold = f.partial; op->n_fold = f.n; op->fold_stride = f.stride; op->fold_bias = f.bias;
    if (fold) *fold = Fold();
    return;
  }
  // the lean instantiation (<= 3 partial sums in registers) unless the pending split is wider
  auto kern = f.n > 3 ? layernorm_kernel<AT, LN_MAXFOLD> : layernorm_kernel<AT, 3>;
  launch_k(ctx, st, "layernorm", kern, dim3(rows), dim3(LN_THREADS), 0, x, g, b, nullptr, out, rows,
           ctx->D, 1, 0, f.partial, f.n, f.stride, f.bias, 1, 1);
  if (fold) *fold = Fold();
}

// LayerNorm with a row mapping (layernorm_kernel: input row (r / in_group) * in_mul + in_off + r % in_group, output row
// r * out_mul); `fold` is NOT cleared: the 'bidirectional' depth pass normalises disjoint row sets with two launches.
template <typename OutT>
static void layernorm_rows(hq_ctx* ctx, cudaStream_t st, const char* tag, float* x, const float* g, const float* b,
                           const float* add, OutT* out, int rows, int in_group, int in_mul, int in_off, int out_mul,
                           const Fold& f) {
  auto kern = f.n > 3 ? layernorm_kernel<OutT, LN_MAXFOLD> : layernorm_kernel<OutT, 3>;
  launch_k(ctx, st, tag, kern, dim3(rows), dim3(LN_THREADS), 0, x, g, b, add, out, rows, ctx->D, in_mul, in_off, f.partial,
           f.n, f.stride, f.bias, in_group, out_mul);
}

// May the decode attention request cached keys BEFORE griddepcontrol.wait?  Yes: run_position orders positions with a
// full dependency, so every earlier position's keys are in place.  (HQ_ATTN_NO_PREFETCH: experiment switch.)
static bool attn_prefetch_ok(const hq_ctx* ctx) { return !ctx->dbg.attn_no_prefetch; }

static int attn_sleep_ns(const hq_ctx* ctx) { return ctx->dbg.attn_sleep; }

// Launch plan of attention_decode_kernel for this model: head groups per image, keys per ring stage, dynamic smem.
template <typename AT>
static bool attn_decode_plan(const hq_ctx* ctx, int* CH, int* hpc, int* groups, size_t* smem) {
  const int g = attn_groups(ctx, ctx->nh);
  if (g <= 0) return false;
  *groups = g;
  *hpc = ctx->nh / g;
  const int row_bytes = *hpc * 64 * static_cast<int>(sizeof(AT));
  int ch = (6144 / row_bytes) / 4 * 4;          // ~6 KB per stage
  if (ch < 4) ch = 4;
  if (ch > 16) ch = 16;
  *CH = ch;
  *smem = static_cast<size_t>(ATTD_STAGES) * ch * row_bytes + static_cast<size_t>(*hpc) * ATT_MAX_KEYS * 4 +
          2 * ATTD_STAGES * 8 + 128;
  return *smem <= 64 * 1024;
}

// Launch plan of attention_decode_mma_kernel (2-byte engines): ring stages of one 8-key K tile + one 8-value V tile (hpc KB each);
// grid = resident CTAs (registers allow four 7-warp CTAs per SM; each takes one item, then tickets), capped by the
// number of items.
static bool attn_mma_plan(const hq_ctx* ctx, int groups, int hpc, int n_items, int* stages, size_t* smem, int* grid) {
  if (ctx->dbg.attn_scalar || !ctx->half || ctx->num_sms <= 0 || !ctx->kv_maps) return false;
  const size_t stage = static_cast<size_t>(2 * ATTM_CH) * hpc * 128;     // K tile + V tile
  // Two stages (24 KB for 6 heads): measured equal end to end to a 4-deep ring and ~1 us faster per launch in the loop
  // (profiles/r1_attn_sweep.txt) - requests beyond the bandwidth-delay product only lengthen every request's latency,
  // and a 27 KB CTA still fits next to a resident GEMM CTA, so its prefetch can start under the QKV GEMM (PDL).
  int st = 2;
  if (ctx->dbg.attm_stages) st = ctx->dbg.attm_stages;            // experiments
  if (st < 2) st = 2;
  if (st > ATTM_MAXSTAGES) st = ATTM_MAXSTAGES;
  const size_t bytes = 1024 /*tile alignment*/ + st * stage + 2 * static_cast<size_t>(hpc) * 128 +
                       static_cast<size_t>(hpc) * 64 * 4 + (2 * ATTM_MAXSTAGES + 4) * 8 + 16;
  if (bytes > 112 * 1024) return false;
  int per_sm = static_cast<int>((227 * 1024) / (bytes + 1024));
  const int by_threads = 2048 / ((hpc + 1) * 32);
  if (per_sm > by_threads) per_sm = by_threads;
  const int by_regs = 65536 / ((hpc + 1) * 32 * 72);              // 72 registers per thread (ptxas)
  if (by_regs >= 1 && per_sm > by_regs) per_sm = by_regs;
  if (ctx->dbg.attm_per_sm > 0 && ctx->dbg.attm_per_sm < per_sm) per_sm = ctx->dbg.attm_per_sm;   // experiments
  if (per_sm < 1) per_sm = 1;
  (void)groups;
  *stages = st;
  *smem = bytes;
  const int cap = ctx->num_sms * per_sm;
  *grid = n_items < cap ? n_items : cap;
  return true;
}

template <typename AT>
static void launch_attn_mma(hq_ctx* ctx, cudaStream_t st, const AT* q, const AT* K, AT* out, int t_stride, int n_keys,
                            int hpc, int groups, int n_items, int stages, int grid, size_t smem) {
  // K (and V, at the same offset in its own cache) as a row offset into the cache-wide tensor maps
  const int row_base = static_cast<int>((K - static_cast<const AT*>(ctx->kc)) / ctx->D);
  launch_k(ctx, st, "attention_decode", attention_decode_mma_kernel<AT>, dim3(grid), dim3((hpc + 1) * 32), smem, ctx->kmap, ctx->vmap,
           row_base, q, out, ctx->D, t_stride, n_keys, hpc, groups, n_items, attn_prefetch_ok(ctx) ? stages : -stages,
           ctx->att_sched);
}
template <>
void launch_attn_mma<float>(hq_ctx*, cudaStream_t, const float*, const float*, float*, int, int, int, int, int, int, int, size_t) {}

template <typename AT>
static void attention(hq_ctx* ctx, cudaStream_t st, const AT* q, const AT* K, const AT* V, AT* out, int M, int Tq,
                      int t_stride, int kbase, int causal) {
  int CH = 0, hpc = 0, groups = 0;
  size_t smem = 0;
  if (ctx->recording && std::is_same<AT, bf16>::value && !causal && kbase <= ATT_DEPTH_KEYS && Tq == 4) {
    ChainOp* op = chain_push(ctx, CH_OP_ATTN4, "attention_depth4");
    op->q = reinterpret_cast<const bf16*>(q); op->kc = reinterpret_cast<const bf16*>(K);
    op->vc = reinterpret_cast<const bf16*>(V); op->att = reinterpret_cast<bf16*>(out);
    op->B = M / 4; op->n_heads = ctx->nh; op->D = ctx->D; op->t_stride = t_stride; op->n_keys = kbase;
    return;
  }
  // any other attention is a kernel of its own: the ops recorded so far go out first, recording resumes after it
  const bool resume = ctx->recording;
  if (resume) chain_flush(ctx, st);
  struct Resume { hq_ctx* c; bool on; ~Resume() { c->recording = on; } } resume_guard{ctx, resume};
  ctx->recording = false;
  if constexpr (sizeof(AT) == 2) {
    if (ctx->prefix_pass && causal && kbase == 0 && Tq <= ATT_MAX_KEYS) {
      // image-completion prefix pass: one CTA per (image, head), K / V staged once, tensor-core QK^T and PV
      launch_k(ctx, st, "attention_prefix", attention_prefix_kernel<AT>, dim3((M / Tq) * ctx->nh), dim3(256), 0, q, K, V, out,
               ctx->nh, ctx->D, Tq, t_stride);
      return;
    }
  }
  if (Tq == 1 && !causal && !ctx->dbg.attn_generic && attn_decode_plan<AT>(ctx, &CH, &hpc, &groups, &smem)) {
    // spatial decode: (image, head group) work items, K/V streamed through shared memory by bulk async copies
    if (ctx->tracing) ctx->tag_suffix = ":t" + std::to_string(kbase) + ":B" + std::to_string(M);
    int stages = 0, grid = 0;
    size_t smem2 = 0;
    // the tensor maps describe ctx->kc / ctx->vc: the TMA kernel needs K and V at the same offset inside them
    const ptrdiff_t koff = reinterpret_cast<const char*>(K) - static_cast<const char*>(ctx->kc);
    const ptrdiff_t kv_bytes = static_cast<ptrdiff_t>(ctx->L) * ctx->max_batch * ctx->Tc * ctx->D * static_cast<ptrdiff_t>(ctx->wsize);
    const bool in_cache = ctx->kc != nullptr && koff >= 0 && (koff < kv_bytes || ctx->L == 0) &&
                          koff == reinterpret_cast<const char*>(V) - static_cast<const char*>(ctx->vc);
    if (sizeof(AT) == 2 && in_cache && attn_mma_plan(ctx, groups, hpc, M * groups, &stages, &smem2, &grid)) {
      launch_attn_mma<AT>(ctx, st, q, K, out, t_stride, kbase, hpc, groups, M * groups, stages, grid, smem2);
      return;
    }
    launch_k(ctx, st, "attention_decode", attention_decode_kernel<AT>, dim3(M * groups), dim3((hpc + 1) * 32), smem, q, K, V,
             out, ctx->D, t_stride, kbase, CH, hpc, groups, attn_prefetch_ok(ctx) ? attn_sleep_ns(ctx) : -1);
    return;
  }
  const int items = M * ctx->nh;
  if (!causal && kbase <= ATT_DEPTH_KEYS && Tq == 4 && !ctx->dbg.attn_fewkeys_old) {
    // the parallel depth pass: one warp per (image, head) serves the image's four queries
    const int warps = (M / 4) * ctx->nh;
    launch_k(ctx, st, "attention_depth4", attention_depth4_kernel<AT>, dim3((warps + ATT_WARPS - 1) / ATT_WARPS),
             dim3(ATT_WARPS * 32), 0, q, K, V, out, M / 4, ctx->nh, ctx->D, t_stride, kbase);
    return;
  }
  if (!causal && kbase <= 8) {
    launch_k(ctx, st, "attention_fewkeys", attention_fewkeys_kernel<AT>, dim3((items + ATT_WARPS - 1) / ATT_WARPS),
             dim3(ATT_WARPS * 32), 0, q, K, V, out, M, ctx->nh, ctx->D, Tq, t_stride, kbase);
    return;
  }
  launch_k(ctx, st, "attention_generic", attention_kernel<AT>, dim3((items + ATT_WARPS - 1) / ATT_WARPS),
           dim3(ATT_WARPS * 32), 0, q, K, V, out, M, ctx->nh, ctx->D, Tq, t_stride, kbase, causal);
}

static void launch_sample(hq_ctx* ctx, cudaStream_t st, const SampleArgs& a) {
  if (a.V <= 256 * SMP_IPT) launch_k(ctx, st, "sample", sample_kernel<256>, dim3(a.R), dim3(256), 0, a);
  else launch_k(ctx, st, "sample", sample_kernel<1024>, dim3(a.R), dim3(1024), 0, a);
}

// One transformer block (layers.py:324-328 / 371-375) on residual stream `x` [M, D].
//   mode 0: spatial decode / prefill  - q, k, v; attention over the spatial cache
//   mode 1: depth pass 0              - k, v only (softmax over one key == identity, a = v)
//   mode 2: depth pass 1              - q, k, v; 4 queries over the 5 depth keys
template <typename AT>
static void gemm_fc2_split(hq_ctx* ctx, cudaStream_t st, const ABuf& A, const Weight& W, int M, int N, int K, int splits,
                           int bn, AT*) {
  EpiParams<AT> e;
  memset(&e, 0, sizeof(e));
  e.outf = ctx->splitk_ws; e.ldo = N; e.split_stride = static_cast<size_t>(ctx->ws_rows) * N;
  ctx->gemm_tag_override = "gemm_resid";
  gemm_tc<EPI_F32, AT>(ctx, st, A.map, A.have3 ? &A.map3 : nullptr, W.map, W.mapp, 0, M, N, K, e, splits, bn, A.map_idx, W.map_idx);
}
template <>
void gemm_fc2_split<float>(hq_ctx*, cudaStream_t, const ABuf&, const Weight&, int, int, int, int, int, float*) {}

// Residual GEMMs (proj [D, D], fc2 [D, 4D]): the narrowest outputs of a block (few CTA pairs) and, for fc2, the longest
// serial K loop.  The K range is cut in up to LN_MAXFOLD slices; the slices write fp32 partial sums that the next
// LayerNorm adds in a fixed order (deterministic).  Same cost model as pick_pair_bn.
struct Fc2Plan { int bn, splits; };

// Split factor of a residual GEMM as a function of its weight shape and of the call site's rows per image (1: spatial
// step / depth pass 0, 4: depth pass 1, T0: text prefill) only - the cost model evaluated at the reference batch of 256
// images, never at the actual batch.  The K slices and the order in which the LayerNorm adds their partial sums fix how
// every output element is rounded; tile widths and kernels (pair / single CTA) do not.  A split that does not depend on
// the batch therefore makes a row's result independent of the batch it sits in - and of how a batch is sharded over GPUs.
static int resid_splits(const hq_ctx* ctx, int N, int K, int rows_per_image) {
  static const int cand[6] = {256, 192, 128, 96, 64, 32};
  const int kb = K / 64;
  // At most 3 slices where 3 divides the k-blocks (every D = 1536 model): measured on the final kernels with the factor
  // pinned for all residual GEMMs (profiles/r2_splitk_final.txt), 3 beats the model's 6 for fc2 at 256 rows end to end
  // (3 482 vs 3 459 images/s) - half the fp32 partial bytes, one epilogue chunk per warp, and the LayerNorm behind it is the
  // 3-fold instantiation (112 instead of 152 registers: more of the next GEMM's CTAs become resident next to it).
  const int max_splits = ctx->dbg.max_splitk > 0 ? ctx->dbg.max_splitk : (kb % 3 == 0 ? 3 : LN_MAXFOLD);
  int best = 1;
  double best_cost = 1e30;
  for (int bn : cand) {
    if (N % bn != 0) continue;
    for (int s = 1; s <= max_splits && s <= LN_MAXFOLD; ++s) {
      if (kb % s != 0) continue;
      const double cost = pair_gemm_cost(256 * (rows_per_image < 1 ? 1 : rows_per_image), N, K, bn, s);
      if (cost < best_cost) {
        best_cost = cost;
        best = s;
      }
    }
  }
  return best;
}

// Tile width for this M given the split (bn = 0: the single-CTA kernel, M <= 128, K slices on grid.z).
static Fc2Plan pick_resid_plan(const hq_ctx* ctx, int M, int N, int K, int rows_per_image) {
  Fc2Plan best{0, 1};
  if (!ctx->half || N % 64 != 0 || K % 64 != 0 || ctx->dbg.no_splitk) return best;
  static const int cand[6] = {256, 192, 128, 96, 64, 32};
  const int kb = K / 64;
  int s = resid_splits(ctx, N, K, rows_per_image);
  {
    const int v = ctx->dbg.force_splitk;                  // tests: pin the split factor
    if (v >= 1 && v <= LN_MAXFOLD && kb % v == 0) s = v;
  }
  best.splits = s;
  if (M <= 128) return best;
  double best_cost = 1e30;
  for (int bn : cand) {
    if (N % bn != 0) continue;
    const double cost = pair_gemm_cost(M, N, K, bn, s);
    if (cost < best_cost) {
      best_cost = cost;
      best.bn = bn;
    }
  }
  return best;
}

// x += A W^T + bias.  Either in the GEMM epilogue, or (split-K) as fp32 partial sums that the next LayerNorm on this
// residual stream folds in; `fold` carries that pending state to the LayerNorm launch.
template <typename AT>
static void gemm_resid(hq_ctx* ctx, cudaStream_t st, const ABuf& A, const Weight& W, const float* bias, float* x, int M,
                       int N, int K, int rows_per_image, Fold* fold) {
  const Fc2Plan plan = pick_resid_plan(ctx, M, N, K, rows_per_image);
  // The image-completion prefix pass never splits: whether M fits the split-K workspace depends on the batch, and a row's
  // rounding must not (its M = B x (T0 + P - 1) GEMMs have tiles enough without slices).
  if (plan.splits > 1 && M <= ctx->ws_rows && !ctx->prefix_pass) {
    gemm_fc2_split(ctx, st, A, W, M, N, K, plan.splits, plan.bn, static_cast<AT*>(nullptr));
    fold->partial = ctx->splitk_ws;
    fold->n = plan.splits;
    fold->stride = static_cast<size_t>(ctx->ws_rows) * N;
    fold->bias = bias;
    return;
  }
  EpiParams<AT> e;
  memset(&e, 0, sizeof(e));
  e.bias = bias; e.x = x;
  gemm_any<EPI_RESID>(ctx, st, A, W, 0, M, N, K, e);
}

template <typename AT>
static void run_block(hq_ctx* ctx, cudaStream_t st, const BlockW& w, float* x, int M, int mode, AT* kdst, AT* vdst,
                      int rpb, int t_stride, int t0, int n_keys_base, int causal, Fold* fold) {
  const int D = ctx->D;
  AT* h = static_cast<AT*>(ctx->h.ptr);
  AT* att = static_cast<AT*>(ctx->att.ptr);
  AT* mlp = static_cast<AT*>(ctx->mlp.ptr);
  AT* q = static_cast<AT*>(ctx->q);
  layernorm_act<AT>(ctx, st, x, w.ln1g, w.ln1b, h, M, fold);
  EpiParams<AT> ep;
  memset(&ep, 0, sizeof(ep));
  ep.q = q; ep.kdst = kdst; ep.vdst = vdst; ep.D = D; ep.rpb = rpb; ep.t_stride = t_stride; ep.t0 = t0;
  if (mode == 1) {
    ep.bias = w.bqkv + D; ep.sec0 = 1; ep.vdup = att;
    gemm_any<EPI_QKV>(ctx, st, ctx->h, w.qkv, D, M, 2 * D, D, ep);
  } else {
    ep.bias = w.bqkv; ep.sec0 = 0; ep.vdup = nullptr;
    if (mode == 0) ctx->rec_flags = CH_F_T0_RT;     // chain op: the cache slot is a per-launch value, not part of the table
    gemm_any<EPI_QKV>(ctx, st, ctx->h, w.qkv, 0, M, 3 * D, D, ep);
    ctx->rec_flags = 0;
    attention<AT>(ctx, st, q, kdst, vdst, att, M, rpb, t_stride, n_keys_base, causal);
  }
  gemm_resid<AT>(ctx, st, ctx->att, w.proj, w.bproj, x, M, D, D, rpb, fold);
  layernorm_act<AT>(ctx, st, x, w.ln2g, w.ln2b, h, M, fold);
  EpiParams<AT> eg;
  memset(&eg, 0, sizeof(eg));
  eg.bias = w.b1; eg.out = mlp;
  gemm_any<EPI_GELU>(ctx, st, ctx->h, w.fc1, 0, M, 4 * D, D, eg);
  gemm_resid<AT>(ctx, st, ctx->mlp, w.fc2, w.b2, x, M, D, 4 * D, rpb, fold);
}

struct RunFlags {
  int forced_top, forced_bot, sos_override, forced_mid;
  int shared_prefix;    // text models: every row has the same prompt - prefill image 0 only, broadcast its cache rows
  int prefix_len;       // image completion: positions < prefix_len are given; run_prefix fills their cache slots
  int prefix_shared;    // ... and every row has the same condition and prefix: the prefix pass runs for image 0 only
  int fuse_mask;        // bit filt_sel (0 top, 1 bottom, 2 middle): that filter pair is (None, None) -> head GEMM draws in its epilogue
  float* logits_out;
};

// Head GEMM of the draw described by `sa` (hierarchical_ar.py:695 / 715).  When the draw has no top-k / top-p cut (the
// measure_throughput protocol) the 2-byte engines sample inside the GEMM epilogue (gemm.cuh: EPI_SAMPLE) and the [rows, V]
// logits are never written; otherwise the logits go to ctx->logits for sample_kernel.  Returns whether it fused.
template <typename AT>
static bool head_gemm(hq_ctx* ctx, cudaStream_t st, const Weight& w, int rows, int V, const SampleArgs& sa, const RunFlags& f) {
  const bool fuse = sizeof(AT) == 2 && !ctx->recording && ((f.fuse_mask >> sa.filt_sel) & 1) && !sa.forced &&
                    sa.logits_out == nullptr && V % 32 == 0;
  EpiParams<AT> e;
  memset(&e, 0, sizeof(e));
  if (fuse) {
    e.sp = sa.sp; e.samp_part = ctx->samp_part; e.temp_sel = sa.temp_sel; e.rows_per_b = sa.rows_per_b; e.slot0 = sa.slot0;
    e.pos = sa.pos;
    ctx->gemm_tag_override = "gemm_head_sample";
    gemm_any<EPI_SAMPLE>(ctx, st, ctx->h, w, 0, rows, V, ctx->D, e);
  } else {
    e.outf = ctx->logits; e.ldo = ctx->Vmax;
    gemm_any<EPI_F32>(ctx, st, ctx->h, w, 0, rows, V, ctx->D, e);
  }
  return fuse;
}

static void draw(hq_ctx* ctx, cudaStream_t st, const SampleArgs& sa, bool fused) {
  if (fused)
    launch_k(ctx, st, "sample_finalize", sample_finalize_kernel, dim3((sa.R + SMPF_WARPS - 1) / SMPF_WARPS), dim3(SMPF_WARPS * 32),
             0, sa, static_cast<const float2*>(ctx->samp_part), sa.V / 32);
  else if (!(sa.forced && sa.logits_out == nullptr))
    launch_sample(ctx, st, sa);
}

// One top position (SURVEY.md 8a-spec): spatial step, depth pass 0, draw top, depth pass 1, draw 4 bottoms.
template <typename AT>
static void run_position(hq_ctx* ctx, cudaStream_t st, int B, int S, int pos, const RunFlags& f) {
  const int D = ctx->D, T0 = ctx->T0, Tc = ctx->Tc;
  const bool txt = ctx->cfg.cond_kind == HQ_COND_TXT;
  const bool prefill = txt && pos == 0;
  const bool shared = prefill && f.shared_prefix && B > 1;
  const int Bp = shared ? 1 : B;                      // images the prefill runs for
  const int M = prefill ? Bp * T0 : B;
  AT* kc = static_cast<AT*>(ctx->kc);
  AT* vc = static_cast<AT*>(ctx->vc);
  AT* kd = static_cast<AT*>(ctx->kd);
  AT* vd = static_cast<AT*>(ctx->vd);
  AT* h = static_cast<AT*>(ctx->h.ptr);
  const size_t lstride = static_cast<size_t>(ctx->max_batch) * Tc * D;
  const size_t dstride = static_cast<size_t>(ctx->max_batch) * 5 * D;

  // one float4 per thread: every gather of a row is in flight at once (a single memory round trip after the codes)
  const int eb = (D / 4 + 31) / 32 * 32 > 1024 ? 1024 : (D / 4 + 31) / 32 * 32;
  Fold fold_x, fold_y;   // split-K partial sums pending on the spatial / depth residual stream
  // ---- K1: input token(s) ----
  // The first kernel of a position is NOT a programmatic dependent: it starts only when the previous position has
  // completed.  Programmatic launches cascade - kernel N+1 may become resident as soon as N has started, N+2 as soon as
  // N+1 has, ... - and with small models (a few CTAs per kernel, < 128 launches per position) the hardware keeps a whole
  // position of not-yet-run kernels resident.  The decode attention requests the keys of EARLIER positions before its
  // griddepcontrol.wait; a barrier per position is what makes "earlier positions are complete" true.  (Found by the
  // asymmetric golden: without it a second run read the previous run's keys, graph + PDL only.)  Cost: ~1 us per position.
  ctx->full_dependency_next = true;
  if (prefill) {
    launch_k(ctx, st, "embed_txt", embed_txt_kernel, dim3(M), dim3(eb), 0, ctx->x, f.sos_override ? ctx->sos_override : nullptr,
             ctx->cond, ctx->E_txt, ctx->P_txt, T0, D);
  } else {
    EmbedArgs ea;
    ea.x = ctx->x; ea.sos_table = ctx->sos_table; ea.sos_override = f.sos_override ? ctx->sos_override : nullptr;
    ea.cond = ctx->cond; ea.E_top = ctx->E_top; ea.E_bot = ctx->E_bot; ea.P_top = ctx->P_top; ea.P_emb = ctx->P_emb;
    ea.codes_top = ctx->codes_top; ea.codes_bot = ctx->codes_bot; ea.D = D; ea.S = S; ea.pos = pos;
    ea.cond_kind = ctx->cfg.cond_kind;
    ea.emb_kind = ctx->cfg.embedding_kind; ea.P_top_h = ctx->P_top_h; ea.P_top_w = ctx->P_top_w; ea.Hpos = ctx->Hpos;
    launch_k(ctx, st, "embed", embed_kernel, dim3(B), dim3(eb), 0, ea);
  }

  // ---- spatial transformer: L blocks over the KV cache ----
  const int tok = (pos == 0) ? 0 : T0 + pos - 1;     // cache slot of this position's (first) token
  // persistent chain kernel: every run of ops between two cache attentions (and the whole depth transformer) is one launch
  const bool chain = std::is_same<AT, bf16>::value && !prefill && chain_enabled(ctx, B);
  if (chain) chain_begin(ctx, tok, pos, S);
  for (int l = 0; l < ctx->L; ++l) {
    if (prefill) run_block<AT>(ctx, st, ctx->blocks[l], ctx->x, M, 0, kc + l * lstride, vc + l * lstride, T0, Tc, 0, 0, 1, &fold_x);
    else run_block<AT>(ctx, st, ctx->blocks[l], ctx->x, M, 0, kc + l * lstride, vc + l * lstride, 1, Tc, tok, tok + 1, 0, &fold_x);
  }
  // ---- hs = ln_f(x) (last prefix row for text), depth start token y = hs + sos_depth ----
  if (ctx->recording) {
    ChainOp* op = chain_push(ctx, CH_OP_LN, "layernorm_f");
    op->flags = CH_F_OUT_F32;
    op->x = ctx->x; op->gamma = ctx->lnf_g; op->beta = ctx->lnf_b; op->add = ctx->sos_depth; op->out = ctx->yd;
    op->rows = B; op->in_mul = 1; op->in_off = 0; op->D = D;
    op->fold = fold_x.partial; op->n_fold = fold_x.n; op->fold_stride = fold_x.stride; op->fold_bias = fold_x.bias;
  } else {
    launch_k(ctx, st, "layernorm_f", fold_x.n > 3 ? layernorm_kernel<float, LN_MAXFOLD> : layernorm_kernel<float, 3>, dim3(B),
             dim3(LN_THREADS), 0, ctx->x, ctx->lnf_g, ctx->lnf_b,
             ctx->sos_depth, ctx->yd, prefill ? Bp : B, D, prefill ? T0 : 1, prefill ? T0 - 1 : 0, fold_x.partial, fold_x.n, fold_x.stride,
             fold_x.bias, 1, ctx->cfg.model_type == HQ_MODEL_BIDIRECTIONAL ? 5 : 1);
  }
  fold_x = Fold();
  if (shared)    // one prompt, B samples: image 0's prefix cache rows (all layers) and depth start token -> images 1..B-1
    launch_k(ctx, st, "broadcast_prefix", broadcast_prefix_kernel<AT>, dim3(T0, ctx->L, B - 1), dim3(256), 0, kc, vc, ctx->yd,
             ctx->max_batch, Tc, D);

  SampleArgs sa;
  memset(&sa, 0, sizeof(sa));
  sa.logits = ctx->logits; sa.ldl = ctx->Vmax; sa.V = ctx->Vt; sa.R = B; sa.rows_per_b = 1; sa.slot0 = 0;
  sa.sp = ctx->d_sp; sa.pos = pos; sa.S = S; sa.dst_codes = ctx->codes_top; sa.dst_w = 1; sa.n_slots = ctx->n_stack;
  sa.forced = f.forced_top; sa.logits_out = f.logits_out; sa.Vmax = ctx->Vmax;
  sa.temp_sel = 0; sa.filt_sel = 0; sa.bot_slot = -1;
  if (ctx->cfg.model_type == HQ_MODEL_TOP2BOT) {
    // ---- 'top2bot' (sampling_depth_baseline, hierarchical_ar.py:565-664): five sequential single-token passes over the
    //      depth blocks with a growing cache [Ld][B][5][D]; pass c writes slot c and attends over slots 0..c ----
    for (int c = 0; c < 5; ++c) {
      if (c >= 1) {
        const float* E = c == 1 ? ctx->E_top_depth : ctx->E_bot_depth;
        const int64_t* codes = c == 1 ? ctx->codes_top + pos : ctx->codes_bot + static_cast<size_t>(pos) * 4 + (c - 2);
        launch_k(ctx, st, "embed_depth_seq", embed_depth_seq_kernel, dim3(B), dim3(eb), 0, ctx->yd, E,
                 static_cast<const float*>(ctx->P_depth + static_cast<size_t>(c - 1) * D), codes, c == 1 ? S : 4 * S, D);
      }
      for (int l = 0; l < ctx->Ld; ++l)
        run_block<AT>(ctx, st, ctx->depths[l], ctx->yd, B, 0, kd + l * dstride, vd + l * dstride, 1, 5, c, c + 1, 0, &fold_y);
      layernorm_act<AT>(ctx, st, ctx->yd, c == 0 ? ctx->lnt_g : ctx->lnb_g, c == 0 ? ctx->lnt_b : ctx->lnb_b, h, B, &fold_y);
      sa.V = c == 0 ? ctx->Vt : ctx->Vb; sa.slot0 = c; sa.bot_slot = c - 1;
      sa.dst_codes = c == 0 ? ctx->codes_top : ctx->codes_bot; sa.dst_w = c == 0 ? 1 : 4;
      sa.temp_sel = sa.filt_sel = c == 0 ? 0 : 1;
      sa.forced = c == 0 ? f.forced_top : f.forced_bot;
      draw(ctx, st, sa, head_gemm<AT>(ctx, st, c == 0 ? ctx->head_top : ctx->head_bot, B, sa.V, sa, f));
    }
    return;
  }
  if (ctx->cfg.model_type == HQ_MODEL_BIDIRECTIONAL) {
    // ---- 'bidirectional' (hierarchical_ar.py:791-878): ONE pass over five tokens per image, [hs + sos_depth (written above
    //      at rows 5b), pos_emb_depth[0..3]], unmasked attention among them; ln_top / head_top on token 0, ln_bot / head_bot on
    //      tokens 1..4.  As in the reference every token is drawn with the bottom filters and softmax_temperature[0]. ----
    launch_k(ctx, st, "depth_pos_rows", depth_pos_rows_kernel, dim3(B), dim3(eb), 0, ctx->yd, static_cast<const float*>(ctx->P_depth), D);
    for (int l = 0; l < ctx->Ld; ++l)
      run_block<AT>(ctx, st, ctx->depths[l], ctx->yd, 5 * B, 2, kd + l * dstride, vd + l * dstride, 5, 5, 0, 5, 0, &fold_y);
    layernorm_rows<AT>(ctx, st, "layernorm", ctx->yd, ctx->lnt_g, ctx->lnt_b, nullptr, h, B, 1, 5, 0, 1, fold_y);
    sa.temp_sel = 0; sa.filt_sel = 1;
    draw(ctx, st, sa, head_gemm<AT>(ctx, st, ctx->head_top, B, ctx->Vt, sa, f));
    layernorm_rows<AT>(ctx, st, "layernorm", ctx->yd, ctx->lnb_g, ctx->lnb_b, nullptr, h, 4 * B, 4, 5, 1, 1, fold_y);
    fold_y = Fold();
    sa.V = ctx->Vb; sa.R = 4 * B; sa.rows_per_b = 4; sa.slot0 = 1; sa.forced = f.forced_bot;
    sa.dst_codes = ctx->codes_bot; sa.dst_w = 4;
    draw(ctx, st, sa, head_gemm<AT>(ctx, st, ctx->head_bot, 4 * B, ctx->Vb, sa, f));
    return;
  }

  // ---- depth pass 0 -> top logits ----
  for (int l = 0; l < ctx->Ld; ++l)
    run_block<AT>(ctx, st, ctx->depths[l], ctx->yd, B, 1, kd + l * dstride, vd + l * dstride, 1, 5, 0, 1, 0, &fold_y);
  layernorm_act<AT>(ctx, st, ctx->yd, ctx->lnt_g, ctx->lnt_b, h, B, &fold_y);
  {
    const bool fused = head_gemm<AT>(ctx, st, ctx->head_top, B, ctx->Vt, sa, f);
    if (chain) chain_end(ctx, st);
    draw(ctx, st, sa, fused);
  }

  // ---- depth pass 1 -> 4 bottom logits ----
  if (chain) {
    chain_begin(ctx, tok, pos, S);
    ChainOp* op = chain_push(ctx, CH_OP_EMBED_DEPTH, "embed_depth");
    op->y = ctx->yd; op->E = ctx->E_top_depth; op->P = ctx->P_depth; op->codes_top = ctx->codes_top; op->B = B; op->D = D;
  } else {
    launch_k(ctx, st, "embed_depth", embed_depth_kernel, dim3(B), dim3(eb), 0, ctx->yd, ctx->E_top_depth, ctx->P_depth,
             ctx->codes_top, S, pos, D);
  }
  for (int l = 0; l < ctx->Ld; ++l)
    run_block<AT>(ctx, st, ctx->depths[l], ctx->yd, 4 * B, 2, kd + l * dstride, vd + l * dstride, 4, 5, 1, 5, 0, &fold_y);
  layernorm_act<AT>(ctx, st, ctx->yd, ctx->lnb_g, ctx->lnb_b, h, 4 * B, &fold_y);
  sa.V = ctx->Vb; sa.R = 4 * B; sa.rows_per_b = 4; sa.slot0 = 1; sa.forced = f.forced_bot;
  sa.temp_sel = 1; sa.filt_sel = 1; sa.dst_codes = ctx->codes_bot; sa.dst_w = 4;
  {
    const bool fused = head_gemm<AT>(ctx, st, ctx->head_bot, 4 * B, ctx->Vb, sa, f);
    if (chain) chain_end(ctx, st);
    draw(ctx, st, sa, fused);
  }
}

// One top position of the 3-level HQTransformer, decoding_type 'parallel-add' (SURVEY.md 8f-2; hqtransformer.py:409-635):
// spatial step over the 21-token stack embedding, then three depth passes - 1 top, 4 middle, 16 bottom tokens - over a
// depth cache of 21 slots (pass 1 sees slots 0..4, pass 2 sees 0..20: the 'parallel' mask of layers.py:154-178), one head
// and one set of (temperature, top-k, top-p) per level, 21 draws (Philox slots 0..20).
template <typename AT>
static void run_position3(hq_ctx* ctx, cudaStream_t st, int B, int S, int pos, const RunFlags& f) {
  const int D = ctx->D, Tc = ctx->Tc;
  AT* kc = static_cast<AT*>(ctx->kc);
  AT* vc = static_cast<AT*>(ctx->vc);
  AT* kd = static_cast<AT*>(ctx->kd);
  AT* vd = static_cast<AT*>(ctx->vd);
  AT* h = static_cast<AT*>(ctx->h.ptr);
  const size_t lstride = static_cast<size_t>(ctx->max_batch) * Tc * D;
  const size_t dstride = static_cast<size_t>(ctx->max_batch) * 21 * D;
  const int eb = (D / 4 + 31) / 32 * 32 > 1024 ? 1024 : (D / 4 + 31) / 32 * 32;
  Fold fold_x, fold_y;
  ctx->full_dependency_next = true;             // one full dependency per position (see run_position)
  Embed3Args ea;
  ea.x = ctx->x; ea.sos_table = ctx->sos_table; ea.sos_override = f.sos_override ? ctx->sos_override : nullptr;
  ea.cond = ctx->cond; ea.E0 = ctx->E_top; ea.E1 = ctx->E_mid; ea.E2 = ctx->E_bot; ea.P_top = ctx->P_top; ea.P_emb = ctx->P_emb;
  ea.codes_top = ctx->codes_top; ea.codes_mid = ctx->codes_mid; ea.codes_bot = ctx->codes_bot;
  ea.D = D; ea.S = S; ea.pos = pos; ea.cond_kind = ctx->cfg.cond_kind;
  launch_k(ctx, st, "embed", embed3_kernel, dim3(B), dim3(eb), 0, ea);
  const int tok = pos;                          // cache slot (no text prefix)
  for (int l = 0; l < ctx->L; ++l)
    run_block<AT>(ctx, st, ctx->blocks[l], ctx->x, B, 0, kc + l * lstride, vc + l * lstride, 1, Tc, tok, tok + 1, 0, &fold_x);
  launch_k(ctx, st, "layernorm_f", fold_x.n > 3 ? layernorm_kernel<float, LN_MAXFOLD> : layernorm_kernel<float, 3>, dim3(B),
           dim3(LN_THREADS), 0, ctx->x, ctx->lnf_g, ctx->lnf_b, ctx->sos_depth, ctx->yd, B, D, 1, 0, fold_x.partial, fold_x.n,
           fold_x.stride, fold_x.bias, 1, 1);
  fold_x = Fold();

  SampleArgs sa;
  memset(&sa, 0, sizeof(sa));
  sa.logits = ctx->logits; sa.ldl = ctx->Vmax; sa.sp = ctx->d_sp; sa.pos = pos; sa.S = S; sa.n_slots = 21;
  sa.logits_out = f.logits_out; sa.Vmax = ctx->Vmax; sa.bot_slot = -1;
  // ---- pass 0: top code (k, v only: softmax over one key is the identity) ----
  for (int l = 0; l < ctx->Ld; ++l)
    run_block<AT>(ctx, st, ctx->depths[l], ctx->yd, B, 1, kd + l * dstride, vd + l * dstride, 1, 21, 0, 1, 0, &fold_y);
  layernorm_act<AT>(ctx, st, ctx->yd, ctx->lnt_g, ctx->lnt_b, h, B, &fold_y);
  sa.V = ctx->Vt; sa.R = B; sa.rows_per_b = 1; sa.slot0 = 0; sa.temp_sel = sa.filt_sel = 0;
  sa.dst_codes = ctx->codes_top; sa.dst_w = 1; sa.forced = f.forced_top;
  draw(ctx, st, sa, head_gemm<AT>(ctx, st, ctx->head_top, B, ctx->Vt, sa, f));
  // ---- pass 1: four middle codes; y_j = E0_depth[c_top] + P1[j]; queries see slots 0..4 ----
  launch_k(ctx, st, "embed_depth", embed_depth_kernel, dim3(B), dim3(eb), 0, ctx->yd, ctx->E_top_depth, ctx->P_depth,
           ctx->codes_top, S, pos, D);
  for (int l = 0; l < ctx->Ld; ++l)
    run_block<AT>(ctx, st, ctx->depths[l], ctx->yd, 4 * B, 2, kd + l * dstride, vd + l * dstride, 4, 21, 1, 5, 0, &fold_y);
  layernorm_act<AT>(ctx, st, ctx->yd, ctx->lnm_g, ctx->lnm_b, h, 4 * B, &fold_y);
  sa.V = ctx->Vm; sa.R = 4 * B; sa.rows_per_b = 4; sa.slot0 = 1; sa.temp_sel = sa.filt_sel = 2;
  sa.dst_codes = ctx->codes_mid; sa.dst_w = 4; sa.forced = f.forced_mid;
  draw(ctx, st, sa, head_gemm<AT>(ctx, st, ctx->head_mid, 4 * B, ctx->Vm, sa, f));
  // ---- pass 2: sixteen bottom codes (raster of the 4x4 cell); queries see slots 0..20 ----
  launch_k(ctx, st, "embed_depth2", embed_depth2_kernel, dim3(B), dim3(eb), 0, ctx->yd, ctx->E_mid_depth, ctx->E_top_depth,
           ctx->P_depth2, ctx->codes_top, ctx->codes_mid, S, pos, D);
  for (int l = 0; l < ctx->Ld; ++l)
    run_block<AT>(ctx, st, ctx->depths[l], ctx->yd, 16 * B, 2, kd + l * dstride, vd + l * dstride, 16, 21, 5, 21, 0, &fold_y);
  layernorm_act<AT>(ctx, st, ctx->yd, ctx->lnb_g, ctx->lnb_b, h, 16 * B, &fold_y);
  sa.V = ctx->Vb; sa.R = 16 * B; sa.rows_per_b = 16; sa.slot0 = 5; sa.temp_sel = sa.filt_sel = 1;
  sa.dst_codes = ctx->codes_bot; sa.dst_w = 16; sa.forced = f.forced_bot;
  draw(ctx, st, sa, head_gemm<AT>(ctx, st, ctx->head_bot, 16 * B, ctx->Vb, sa, f));
}

// Image completion (hq_run_args.prefix_len = P): the spatial KV cache of the given positions 0 .. P - 2 (cache slots
// 0 .. T0 + P - 2) in ONE causal pass over the T0 + P - 1 tokens of every image - the text prefill's shape, large-M GEMMs -
// instead of P steps of the loop.  It depends on the given codes only: no depth pass, ln_f, head or draw.  run_position(P)
// then embeds stack P - 1 into slot T0 + P - 1 as usual and samples on.  The last block stops after its QKV GEMM (its
// attention output and MLP feed nothing).  No chain kernel here, as for the text prefill.  Shared prefix: image 0 only, then
// its cache rows (every layer) are broadcast; the depth start token is computed per row by step P.
template <typename AT>
static void run_prefix(hq_ctx* ctx, cudaStream_t st, int B, int S, const RunFlags& f) {
  const int D = ctx->D, T0 = ctx->T0, Tc = ctx->Tc, L = ctx->L;
  const int N = T0 + f.prefix_len - 1;                 // tokens per image
  const bool shared = f.prefix_shared && B > 1;
  const int M = (shared ? 1 : B) * N;
  AT* kc = static_cast<AT*>(ctx->kc);
  AT* vc = static_cast<AT*>(ctx->vc);
  const size_t lstride = static_cast<size_t>(ctx->max_batch) * Tc * D;
  const int eb = (D / 4 + 31) / 32 * 32 > 1024 ? 1024 : (D / 4 + 31) / 32 * 32;
  // the prefix workspace stands in for the step activations while the pass runs
  std::swap(ctx->h, ctx->pre_h); std::swap(ctx->att, ctx->pre_att); std::swap(ctx->mlp, ctx->pre_mlp); std::swap(ctx->q, ctx->pre_q);
  ctx->full_dependency_next = true;                    // as every position's first kernel (see run_position)
  if (ctx->levels == 3) {
    Embed3Args ea;
    ea.x = ctx->pre_x; ea.sos_table = ctx->sos_table; ea.sos_override = f.sos_override ? ctx->sos_override : nullptr;
    ea.cond = ctx->cond; ea.E0 = ctx->E_top; ea.E1 = ctx->E_mid; ea.E2 = ctx->E_bot; ea.P_top = ctx->P_top; ea.P_emb = ctx->P_emb;
    ea.codes_top = ctx->codes_top; ea.codes_mid = ctx->codes_mid; ea.codes_bot = ctx->codes_bot;
    ea.D = D; ea.S = S; ea.pos = 0; ea.cond_kind = ctx->cfg.cond_kind;
    launch_k(ctx, st, "embed_prefix", embed3_prefix_kernel, dim3(M), dim3(eb), 0, ea, N);
  } else {
    EmbedArgs ea;
    ea.x = ctx->pre_x; ea.sos_table = ctx->sos_table; ea.sos_override = f.sos_override ? ctx->sos_override : nullptr;
    ea.cond = ctx->cond; ea.E_top = ctx->E_top; ea.E_bot = ctx->E_bot; ea.P_top = ctx->P_top; ea.P_emb = ctx->P_emb;
    ea.codes_top = ctx->codes_top; ea.codes_bot = ctx->codes_bot; ea.D = D; ea.S = S; ea.pos = 0;
    ea.cond_kind = ctx->cfg.cond_kind;
    ea.emb_kind = ctx->cfg.embedding_kind; ea.P_top_h = ctx->P_top_h; ea.P_top_w = ctx->P_top_w; ea.Hpos = ctx->Hpos;
    launch_k(ctx, st, "embed_prefix", embed_prefix_kernel, dim3(M), dim3(eb), 0, ea, static_cast<const float*>(ctx->E_txt),
             static_cast<const float*>(ctx->P_txt), T0, N);
  }
  ctx->prefix_pass = true;
  Fold fold;
  for (int l = 0; l + 1 < L; ++l)
    run_block<AT>(ctx, st, ctx->blocks[l], ctx->pre_x, M, 0, kc + l * lstride, vc + l * lstride, N, Tc, 0, 0, 1, &fold);
  {
    const BlockW& w = ctx->blocks[L - 1];
    layernorm_act<AT>(ctx, st, ctx->pre_x, w.ln1g, w.ln1b, static_cast<AT*>(ctx->h.ptr), M, &fold);
    EpiParams<AT> ep;
    memset(&ep, 0, sizeof(ep));
    ep.q = static_cast<AT*>(ctx->q); ep.kdst = kc + (L - 1) * lstride; ep.vdst = vc + (L - 1) * lstride; ep.D = D; ep.rpb = N;
    ep.t_stride = Tc; ep.t0 = 0; ep.bias = w.bqkv; ep.sec0 = 0; ep.vdup = nullptr;
    gemm_any<EPI_QKV>(ctx, st, ctx->h, w.qkv, 0, M, 3 * D, D, ep);
  }
  ctx->prefix_pass = false;
  std::swap(ctx->h, ctx->pre_h); std::swap(ctx->att, ctx->pre_att); std::swap(ctx->mlp, ctx->pre_mlp); std::swap(ctx->q, ctx->pre_q);
  if (shared)    // image 0's N cache rows of every layer -> images 1..B-1 (the kernel's copy of yd row 0 is rewritten by step P)
    launch_k(ctx, st, "broadcast_prefix", broadcast_prefix_kernel<AT>, dim3(N, L, B - 1), dim3(256), 0, kc, vc, ctx->yd,
             ctx->max_batch, Tc, D);
}

static void run_range(hq_ctx* ctx, cudaStream_t st, int B, int S, int p0, int p1, const RunFlags& f) {
  with_act(ctx->prec, [&](auto tag) {
    using AT = decltype(tag);
    if (f.prefix_len > 0) run_prefix<AT>(ctx, st, B, S, f);
    for (int pos = p0 + f.prefix_len; pos < p1; ++pos) {
      if (ctx->levels == 3) run_position3<AT>(ctx, st, B, S, pos, f);
      else run_position<AT>(ctx, st, B, S, pos, f);
    }
  });
}

static int validate_run(hq_ctx* ctx, const hq_run_args* a) {
  if (!ctx || !a) return HQ_ERR_INVALID;
  int rc = hq_params_complete(ctx);
  if (rc) return rc;
  if (a->batch < 1 || a->batch > ctx->max_batch) {
    set_err(ctx, "batch %d outside [1, max_batch=%d]", a->batch, ctx->max_batch);
    return HQ_ERR_INVALID;
  }
  if (a->seq_len < 1 || a->seq_len > ctx->Smax || a->pos_begin < 0 || a->pos_end > a->seq_len || a->pos_begin >= a->pos_end) {
    set_err(ctx, "bad position range [%d, %d) for seq_len %d (max_seq_len %d)", a->pos_begin, a->pos_end, a->seq_len, ctx->Smax);
    return HQ_ERR_INVALID;
  }
  if (!a->codes_top || !a->codes_bot || (ctx->levels == 3 && !a->codes_mid)) {
    set_err(ctx, "codes_top / codes_bot%s must not be null", ctx->levels == 3 ? " / codes_mid" : "");
    return HQ_ERR_INVALID;
  }
  if (a->pos_begin == 0 && !a->sos && !a->cond && ctx->cfg.cond_kind != HQ_COND_UNCOND) {
    set_err(ctx, "conditional model: `cond` (or `sos`) is required at pos_begin == 0");
    return HQ_ERR_INVALID;
  }
  if (a->prefix_len < 0) {
    set_err(ctx, "prefix_len must be >= 0 (got %d)", a->prefix_len);
    return HQ_ERR_INVALID;
  }
  if (a->prefix_len > 0) {
    if (a->pos_begin != 0) {
      set_err(ctx, "prefix_len %d needs pos_begin == 0 (got %d): a completion starts a new batch", a->prefix_len, a->pos_begin);
      return HQ_ERR_INVALID;
    }
    if (a->prefix_len >= a->pos_end) {
      set_err(ctx, "prefix_len %d must be below pos_end %d (at least one position is sampled)", a->prefix_len, a->pos_end);
      return HQ_ERR_INVALID;
    }
    if (ctx->T0 + a->prefix_len - 1 > ATT_MAX_KEYS) {
      set_err(ctx, "prefix_len %d: %d prefix tokens exceed the %d keys of the attention kernels", a->prefix_len,
              ctx->T0 + a->prefix_len - 1, ATT_MAX_KEYS);
      return HQ_ERR_INVALID;
    }
  }
  const hq_sampling_params& s = a->sampling;
  if (!(s.temperature_top > 0.f) || !(s.temperature_bot > 0.f)) {
    set_err(ctx, "softmax temperatures must be > 0 (got %g, %g)", s.temperature_top, s.temperature_bot);
    return HQ_ERR_INVALID;
  }
  return HQ_OK;
}

// The image-completion workspace for `rows` prefix tokens (grown, never shrunk, until hq_reserve_batch).  Graphs captured
// with a prefix point into the buffers being replaced: they go too.  Runs without a prefix never come here.
static int ensure_prefix_ws(hq_ctx* ctx, int rows) {
  if (rows <= ctx->pre_rows) return HQ_OK;
  HQ_CUDA(ctx, cudaDeviceSynchronize());
  for (auto it = ctx->graphs.begin(); it != ctx->graphs.end();) {
    if (it->first.prefix_len > 0) {
      cudaGraphExecDestroy(it->second.exec);
      it = ctx->graphs.erase(it);
    } else {
      ++it;
    }
  }
  free_prefix_ws(ctx);
  ctx->alloc_pre = true;
  struct Guard { hq_ctx* c; ~Guard() { c->alloc_pre = false; } } guard{ctx};
  const int D = ctx->D;
  int rc;
  if ((rc = alloc_abuf(ctx, &ctx->pre_h, rows, D)) || (rc = alloc_abuf(ctx, &ctx->pre_att, rows, D)) ||
      (rc = alloc_abuf(ctx, &ctx->pre_mlp, rows, 4 * D)) ||
      (rc = dev_alloc(ctx, &ctx->pre_q, static_cast<size_t>(rows) * D * ctx->wsize)) ||
      (rc = alloc_f32(ctx, &ctx->pre_x, static_cast<size_t>(rows) * D))) {
    const std::string why = ctx->err;
    cudaGetLastError();
    free_prefix_ws(ctx);
    set_err(ctx, "image-completion workspace of %d rows: %s", rows, why.c_str());
    return rc;
  }
  ctx->pre_rows = rows;
  return HQ_OK;
}

static int run_impl(hq_ctx* ctx, const hq_run_args* a, cudaStream_t st, cudaMemcpyKind in_kind, cudaMemcpyKind out_kind) {
  int rc = validate_run(ctx, a);
  if (rc) return rc;
  HQ_CUDA(ctx, cudaSetDevice(ctx->device));
  const int B = a->batch, S = a->seq_len, D = ctx->D, T0 = ctx->T0, P = a->prefix_len;
  const size_t nt = static_cast<size_t>(B) * S * 8, nb = nt * (ctx->levels == 3 ? 16 : 4), nm = nt * 4;
  const int prefix_shared = P > 0 && a->shared_prefix != 0 && a->sos == nullptr;
  if (P > 0 && (rc = ensure_prefix_ws(ctx, (prefix_shared && B > 1 ? 1 : B) * (T0 + P - 1)))) return rc;

  // ---- stage inputs into ctx-owned buffers (what the captured graph reads) ----
  // pageable source: the runtime stages it before returning, so back-to-back calls cannot race on it
  HQ_CUDA(ctx, cudaMemcpyAsync(ctx->d_sp, &a->sampling, sizeof(hq_sampling_params), cudaMemcpyHostToDevice, st));
  if (a->pos_begin == 0) {
    if (a->cond && ctx->cfg.cond_kind != HQ_COND_UNCOND)
      HQ_CUDA(ctx, cudaMemcpyAsync(ctx->cond, a->cond, static_cast<size_t>(B) * T0 * 8, in_kind, st));
    if (a->sos)
      HQ_CUDA(ctx, cudaMemcpyAsync(ctx->sos_override, a->sos, static_cast<size_t>(B) * T0 * D * 4, in_kind, st));
  }
  if (a->pos_begin > 0 || P > 0) {     // the codes of the earlier positions (a continued batch, or a completion's prefix)
    HQ_CUDA(ctx, cudaMemcpyAsync(ctx->codes_top, a->codes_top, nt, in_kind, st));
    HQ_CUDA(ctx, cudaMemcpyAsync(ctx->codes_bot, a->codes_bot, nb, in_kind, st));
    if (ctx->levels == 3) HQ_CUDA(ctx, cudaMemcpyAsync(ctx->codes_mid, a->codes_mid, nm, in_kind, st));
  }
  if (P == 0) {
    if (a->given_top) HQ_CUDA(ctx, cudaMemcpyAsync(ctx->codes_top, a->given_top, nt, in_kind, st));
    if (a->given_bot) HQ_CUDA(ctx, cudaMemcpyAsync(ctx->codes_bot, a->given_bot, nb, in_kind, st));
    if (ctx->levels == 3 && a->given_mid) HQ_CUDA(ctx, cudaMemcpyAsync(ctx->codes_mid, a->given_mid, nm, in_kind, st));
  } else {
    // forced codes apply at positions >= P only: the prefix keeps the codes just copied in
    auto given_tail = [&](int64_t* dst, const int64_t* src, size_t per_pos) {
      const size_t pitch = static_cast<size_t>(S) * per_pos * 8, off = static_cast<size_t>(P) * per_pos;
      return cudaMemcpy2DAsync(dst + off, pitch, src + off, pitch, pitch - off * 8, B, in_kind, st);
    };
    if (a->given_top) HQ_CUDA(ctx, given_tail(ctx->codes_top, a->given_top, 1));
    if (a->given_bot) HQ_CUDA(ctx, given_tail(ctx->codes_bot, a->given_bot, ctx->levels == 3 ? 16 : 4));
    if (ctx->levels == 3 && a->given_mid) HQ_CUDA(ctx, given_tail(ctx->codes_mid, a->given_mid, 4));
  }

  RunFlags f;
  f.forced_top = a->given_top != nullptr;
  f.forced_bot = a->given_bot != nullptr;
  f.forced_mid = ctx->levels == 3 && a->given_mid != nullptr;
  f.shared_prefix = P == 0 && a->shared_prefix != 0 && ctx->cfg.cond_kind == HQ_COND_TXT && a->sos == nullptr &&
                    ctx->cfg.model_type != HQ_MODEL_BIDIRECTIONAL;
  f.prefix_len = P;
  f.prefix_shared = prefix_shared;
  f.sos_override = a->sos != nullptr;
  f.fuse_mask = 0;
  if (ctx->cfg.fuse_head_sampler && ctx->half) {
    const hq_sampling_params& q = a->sampling;
    auto none = [](int k, float p2, int V) { return (k <= 0 || k >= V) && !(p2 > 0.f && p2 < 1.f); };
    if (none(q.top_k_top, q.top_p_top, ctx->Vt)) f.fuse_mask |= 1;
    if (none(q.top_k_bot, q.top_p_bot, ctx->Vb)) f.fuse_mask |= 2;
    if (ctx->levels == 3 && none(q.top_k_mid, q.top_p_mid, ctx->Vm)) f.fuse_mask |= 4;
  }
  f.logits_out = nullptr;
  float* dev_logits = nullptr;
  const size_t nlog = static_cast<size_t>(B) * S * ctx->n_stack * ctx->Vmax * 4;
  if (a->logits) {
    if (out_kind == cudaMemcpyDeviceToHost) {
      HQ_CUDA(ctx, cudaMalloc(reinterpret_cast<void**>(&dev_logits), nlog));
      HQ_CUDA(ctx, cudaMemsetAsync(dev_logits, 0, nlog, st));
      f.logits_out = dev_logits;
    } else {
      f.logits_out = a->logits;
    }
  }

  ctx->launches = 0;
  ctx->launch_err = cudaSuccess;
  const bool use_graph = ctx->cfg.use_cuda_graph && f.logits_out == nullptr;
  // persistent chain kernel: its grid-barrier counter restarts at zero with every run (the captured launches carry the
  // absolute arrival counts they start from), and the op tables are built by a planning pass BEFORE any capture
  ctx->chain_mode = hq_ctx::CHAIN_OFF;
  ctx->recording = false;
  ctx->chain_epoch = 0;
  ctx->chain_launches_run = 0;
  if (ctx->chain_ok) {
    ctx->chain_mode = hq_ctx::CHAIN_RUN;
    if (chain_enabled(ctx, B)) HQ_CUDA(ctx, cudaMemsetAsync(ctx->d_chain_bar, 0, 8, st));
    else ctx->chain_mode = hq_ctx::CHAIN_OFF;
  }
  auto plan_chains = [&]() {
    if (ctx->chain_mode != hq_ctx::CHAIN_RUN) return;
    ctx->chain_mode = hq_ctx::CHAIN_PLAN;
    run_range(ctx, st, B, S, a->pos_begin, a->pos_end, f);
    if (ctx->launch_err == cudaErrorMemoryAllocation) {
      // op-table arena full (many distinct batch sizes): drop every table and every graph that points at one, re-plan
      cudaDeviceSynchronize();
      for (auto& kv : ctx->graphs) cudaGraphExecDestroy(kv.second.exec);
      ctx->graphs.clear();
      ctx->chain_index.clear();
      ctx->ops_used = 0;
      ctx->launch_err = cudaSuccess;
      ctx->recording = false;
      run_range(ctx, st, B, S, a->pos_begin, a->pos_end, f);
    }
    ctx->chain_mode = hq_ctx::CHAIN_RUN;
    ctx->recording = false;
    ctx->chain_epoch = 0;
    ctx->chain_launches_run = 0;
    ctx->launches = 0;
  };
  if (use_graph) {
    GraphKey key{B, S, a->pos_begin, a->pos_end, f.forced_top,
                 f.forced_bot | (f.forced_mid << 1) | (f.shared_prefix << 2) | (f.fuse_mask << 3) | (f.prefix_shared << 6), f.sos_override,
                 ctx->tracing ? 1 : 0, P};
    auto it = ctx->graphs.find(key);
    if (it == ctx->graphs.end()) {
      plan_chains();
      if (ctx->launch_err != cudaSuccess) {
        set_err(ctx, "chain planning failed: %s", cudaGetErrorString(ctx->launch_err));
        return HQ_ERR_CUDA;
      }
      cudaGraph_t graph = nullptr;
      HQ_CUDA(ctx, cudaStreamBeginCapture(ctx->own_stream, cudaStreamCaptureModeThreadLocal));
      run_range(ctx, ctx->own_stream, B, S, a->pos_begin, a->pos_end, f);
      cudaError_t ce = cudaStreamEndCapture(ctx->own_stream, &graph);
      if (ce != cudaSuccess || ctx->launch_err != cudaSuccess) {
        set_err(ctx, "graph capture failed: %s / %s", cudaGetErrorString(ce), cudaGetErrorString(ctx->launch_err));
        if (graph) cudaGraphDestroy(graph);
        return HQ_ERR_CUDA;
      }
      cudaGraphExec_t exec = nullptr;
      cudaError_t ie = cudaGraphInstantiate(&exec, graph, 0);
      cudaGraphDestroy(graph);
      if (ie != cudaSuccess) {
        set_err(ctx, "cudaGraphInstantiate failed: %s", cudaGetErrorString(ie));
        return HQ_ERR_CUDA;
      }
      if (ctx->graphs.size() >= hq_ctx::kMaxGraphs) {     // evict the least recently used graph
        auto victim = ctx->graphs.begin();
        for (auto g = ctx->graphs.begin(); g != ctx->graphs.end(); ++g)
          if (g->second.stamp < victim->second.stamp) victim = g;
        // a replay of the victim may still be in flight on the caller's stream
        HQ_CUDA(ctx, cudaStreamSynchronize(st));
        cudaGraphExecDestroy(victim->second.exec);
        ctx->graphs.erase(victim);
      }
      it = ctx->graphs.emplace(key, hq_ctx::GraphEntry{exec, ctx->launches, 0}).first;
    }
    it->second.stamp = ++ctx->graph_clock;
    HQ_CUDA(ctx, cudaGraphLaunch(it->second.exec, st));
    ctx->last_launches = it->second.launches;
  } else {
    plan_chains();
    run_range(ctx, st, B, S, a->pos_begin, a->pos_end, f);
    ctx->last_launches = ctx->launches;
    if (ctx->launch_err != cudaSuccess) {
      set_err(ctx, "kernel launch failed: %s", cudaGetErrorString(ctx->launch_err));
      if (dev_logits) cudaFree(dev_logits);
      return HQ_ERR_CUDA;
    }
  }

  HQ_CUDA(ctx, cudaMemcpyAsync(a->codes_top, ctx->codes_top, nt, out_kind, st));
  HQ_CUDA(ctx, cudaMemcpyAsync(a->codes_bot, ctx->codes_bot, nb, out_kind, st));
  if (ctx->levels == 3) HQ_CUDA(ctx, cudaMemcpyAsync(a->codes_mid, ctx->codes_mid, nm, out_kind, st));
  if (dev_logits) {
    if (P > 0) {    // positions >= P only: the caller's prefix rows stay untouched
      const size_t row = nlog / B, off = row / S * P;
      HQ_CUDA(ctx, cudaMemcpy2DAsync(reinterpret_cast<char*>(a->logits) + off, row, reinterpret_cast<const char*>(dev_logits) + off,
                                     row, row - off, B, cudaMemcpyDeviceToHost, st));
    } else {
      HQ_CUDA(ctx, cudaMemcpyAsync(a->logits, dev_logits, nlog, cudaMemcpyDeviceToHost, st));
    }
    HQ_CUDA(ctx, cudaStreamSynchronize(st));
    cudaFree(dev_logits);
  }
  return HQ_OK;
}

extern "C" int hq_run(hq_ctx* ctx, const hq_run_args* args, void* stream) {
  return run_impl(ctx, args, static_cast<cudaStream_t>(stream), cudaMemcpyDeviceToDevice, cudaMemcpyDeviceToDevice);
}

extern "C" int hq_run_host(hq_ctx* ctx, const hq_run_args* args) {
  if (!ctx) return HQ_ERR_INVALID;
  int rc = run_impl(ctx, args, ctx->own_stream, cudaMemcpyHostToDevice, cudaMemcpyDeviceToHost);
  if (rc) return rc;
  HQ_CUDA(ctx, cudaStreamSynchronize(ctx->own_stream));
  return HQ_OK;
}

// ------------------------------------------------------------------------------------------------
// test / measurement hooks
// ------------------------------------------------------------------------------------------------
extern "C" int hq_debug_attention(int prec, const void* q, const void* K, const void* V, void* out, int B, int n_heads,
                                  int t_stride, int n_keys, int variant, void* stream) {
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (B < 1 || n_heads < 1 || n_keys < 1 || n_keys > t_stride || n_keys > ATT_MAX_KEYS || !q || !K || !V || !out) {
    set_err(nullptr, "hq_debug_attention: bad argument");
    return HQ_ERR_INVALID;
  }
  hq_ctx tmp;   // launch bookkeeping + the fields attention() reads
  int dev = 0;
  HQ_CUDA(nullptr, cudaGetDevice(&dev));
  int rc = check_device(&tmp, dev);
  if (rc) return rc;
  tmp.prec = (prec == HQ_PREC_BF16 || prec == HQ_PREC_F16) ? prec : HQ_PREC_FP32;
  tmp.half = tmp.prec != HQ_PREC_FP32;
  tmp.D = n_heads * 64;
  tmp.nh = n_heads;
  HQ_CUDA(nullptr, cudaDeviceGetAttribute(&tmp.num_sms, cudaDevAttrMultiProcessorCount, dev));
  if ((rc = set_attn_attrs(&tmp))) return rc;
  HQ_CUDA(nullptr, cudaMalloc(reinterpret_cast<void**>(&tmp.att_sched), 16));
  cudaMemsetAsync(tmp.att_sched, 0, 16, st);
  if (tmp.half && variant != 1) {
    const int groups = attn_groups(&tmp, n_heads);
    tmp.kc = const_cast<void*>(K);
    tmp.vc = const_cast<void*>(V);
    if ((rc = get_encode_fn(&tmp, &tmp.encode)) == HQ_OK && groups > 0 &&
        (rc = make_kv_map(&tmp, &tmp.kmap, K, n_heads, static_cast<uint64_t>(B) * t_stride, n_heads / groups)) == HQ_OK &&
        (rc = make_kv_map(&tmp, &tmp.vmap, V, n_heads, static_cast<uint64_t>(B) * t_stride, n_heads / groups)) == HQ_OK)
      tmp.kv_maps = true;
    if (rc) {
      cudaFree(tmp.att_sched);
      set_err(nullptr, "hq_debug_attention: %s", tmp.err.c_str());
      return rc;
    }
  }
  if (variant == 1) tmp.dbg.attn_scalar = 1;
  with_act(tmp.prec, [&](auto tag) {
    using AT = decltype(tag);
    attention<AT>(&tmp, st, static_cast<const AT*>(q), static_cast<const AT*>(K), static_cast<const AT*>(V), static_cast<AT*>(out),
                  B, 1, t_stride, n_keys, 0);
  });
  cudaError_t e = cudaStreamSynchronize(st);
  cudaFree(tmp.att_sched);
  if (e == cudaSuccess) e = tmp.launch_err;
  if (e != cudaSuccess) {
    set_err(nullptr, "hq_debug_attention: %s", cudaGetErrorString(e));
    return HQ_ERR_CUDA;
  }
  return HQ_OK;
}

extern "C" int hq_debug_attention_prefix(int prec, const void* q, const void* K, const void* V, void* out, int B, int n_heads,
                                         int t_stride, int n_q, int variant, void* stream) {
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (B < 1 || n_heads < 1 || n_q < 1 || n_q > t_stride || n_q > ATT_MAX_KEYS || !q || !K || !V || !out) {
    set_err(nullptr, "hq_debug_attention_prefix: bad argument");
    return HQ_ERR_INVALID;
  }
  hq_ctx tmp;   // launch bookkeeping + the fields attention() reads
  int dev = 0;
  HQ_CUDA(nullptr, cudaGetDevice(&dev));
  int rc = check_device(&tmp, dev);
  if (rc) return rc;
  tmp.prec = (prec == HQ_PREC_BF16 || prec == HQ_PREC_F16) ? prec : HQ_PREC_FP32;
  tmp.half = tmp.prec != HQ_PREC_FP32;
  tmp.D = n_heads * 64;
  tmp.nh = n_heads;
  tmp.prefix_pass = variant != 1;
  with_act(tmp.prec, [&](auto tag) {
    using AT = decltype(tag);
    attention<AT>(&tmp, st, static_cast<const AT*>(q), static_cast<const AT*>(K), static_cast<const AT*>(V), static_cast<AT*>(out),
                  B * n_q, n_q, t_stride, 0, 1);
  });
  cudaError_t e = cudaStreamSynchronize(st);
  if (e == cudaSuccess) e = tmp.launch_err;
  if (e != cudaSuccess) {
    set_err(nullptr, "hq_debug_attention_prefix: %s", cudaGetErrorString(e));
    return HQ_ERR_CUDA;
  }
  return HQ_OK;
}

extern "C" int hq_debug_gemm(int prec, const void* A, const void* W, float* C, int M, int N, int K, int tile,
                             void* stream) {
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  hq_ctx tmp;   // only used for error text + launch bookkeeping
  if (M < 1 || N < 8 || K < 16) {
    set_err(nullptr, "hq_debug_gemm: bad shape");
    return HQ_ERR_INVALID;
  }
  if (prec == HQ_PREC_FP32) {
    if (K % 16 != 0 || N % 8 != 0) {
      set_err(nullptr, "hq_debug_gemm(fp32): K %% 16 and N %% 8 must be 0");
      return HQ_ERR_INVALID;
    }
    EpiParams<float> e;
    memset(&e, 0, sizeof(e));
    e.outf = C; e.ldo = N;
    gemm_f32<EPI_F32>(&tmp, st, static_cast<const float*>(A), static_cast<const float*>(W), M, N, K, e);
  } else {
    if (prec != HQ_PREC_BF16 && prec != HQ_PREC_F16) {
      set_err(nullptr, "hq_debug_gemm: unknown precision %d", prec);
      return HQ_ERR_INVALID;
    }
    if (K % 64 != 0 || N % 64 != 0) {
      set_err(nullptr, "hq_debug_gemm(bf16 / fp16): K %% 64 and N %% 64 must be 0");
      return HQ_ERR_INVALID;
    }
    tmp.prec = prec;
    int dev = 0;
    HQ_CUDA(nullptr, cudaGetDevice(&dev));
    int rc = check_device(&tmp, dev);
    if (rc == HQ_OK) rc = get_encode_fn(&tmp, &tmp.encode);
    if (rc == HQ_OK) rc = set_gemm_attrs_for(&tmp);
    // A rows are padded to the 128-row tile by a zero-filled staging copy so that the TMA box never leaves the tensor
    const int Mp = (M + 127) / 128 * 128;
    void* Ap = nullptr;
    if (rc == HQ_OK) {
      HQ_CUDA(nullptr, cudaMalloc(&Ap, static_cast<size_t>(Mp) * K * 2));
      cudaMemsetAsync(Ap, 0, static_cast<size_t>(Mp) * K * 2, st);
      cudaMemcpyAsync(Ap, A, static_cast<size_t>(M) * K * 2, cudaMemcpyDeviceToDevice, st);
    }
    CUtensorMap mA, mA3, mW;
    PairMaps mWp;
    if (rc == HQ_OK) rc = make_map(&tmp, &mA, Ap, Mp, K, 128);
    if (rc == HQ_OK && K >= 128) rc = make_map3(&tmp, &mA3, Ap, Mp, K, 128, 2);
    if (rc == HQ_OK) rc = make_map(&tmp, &mW, const_cast<void*>(W), N, K, 64);
    if (rc == HQ_OK) rc = make_pair_maps(&tmp, &mWp, const_cast<void*>(W), N, K);
    if (rc == HQ_OK) {
      tmp.dbg.force_bn = tile;
      with_act(prec, [&](auto tag) {
        using AT = decltype(tag);
        if constexpr (sizeof(AT) == 2) {
          EpiParams<AT> e;
          memset(&e, 0, sizeof(e));
          e.outf = C; e.ldo = N;
          gemm_tc<EPI_F32, AT>(&tmp, st, mA, K >= 128 ? &mA3 : nullptr, mW, mWp, 0, M, N, K, e);
        }
      });
    }
    cudaError_t se = cudaStreamSynchronize(st);
    if (Ap) cudaFree(Ap);
    if (rc != HQ_OK) {
      g_last_error = tmp.err;
      return rc;
    }
    if (se != cudaSuccess) {
      set_err(nullptr, "hq_debug_gemm: %s", cudaGetErrorString(se));
      return HQ_ERR_CUDA;
    }
  }
  if (tmp.launch_err != cudaSuccess) {
    set_err(nullptr, "hq_debug_gemm launch failed: %s", cudaGetErrorString(tmp.launch_err));
    return HQ_ERR_CUDA;
  }
  return HQ_OK;
}

// The fused epilogue of one hq_debug_gemm_epi launch as the GEMM kernels take it.
template <typename AT>
static EpiParams<AT> debug_epi_params(const hq_debug_epi* d) {
  EpiParams<AT> ep;
  memset(&ep, 0, sizeof(ep));
  ep.bias = d->bias;
  ep.q = static_cast<AT*>(d->q); ep.kdst = static_cast<AT*>(d->kdst); ep.vdst = static_cast<AT*>(d->vdst);
  ep.vdup = static_cast<AT*>(d->vdup);
  ep.D = d->D; ep.sec0 = d->sec0; ep.rpb = d->rpb; ep.t_stride = d->t_stride; ep.t0 = d->t0;
  ep.x = d->x;
  ep.out = static_cast<AT*>(d->out);
  ep.outf = d->outf; ep.ldo = d->ldo; ep.split_stride = static_cast<size_t>(d->split_stride);
  return ep;
}

static const char* debug_epi_invalid(int prec, int w_rows, int M, int N, int K, const hq_debug_epi* d) {
  if (prec != HQ_PREC_BF16 && prec != HQ_PREC_F16 && prec != HQ_PREC_FP32) return "unknown precision";
  if (M < 1 || N < 32 || N % 32 != 0 || K < 64 || K % 64 != 0) return "shape: need M >= 1, N % 32 == 0, K % 64 == 0";
  if (d->w_row_off < 0 || w_rows < d->w_row_off + N) return "W needs w_rows >= w_row_off + N rows";
  if (d->epi < EPI_QKV || d->epi > EPI_F32) return "epi must be QKV, RESID, GELU or F32";
  if (d->splits < 1 || d->splits > LN_MAXFOLD || (K / 64) % d->splits != 0) return "splits must divide K / 64 (1..6)";
  if (d->splits > 1 && d->epi != EPI_F32) return "split-K is an EPI_F32 launch only";
  if (prec == HQ_PREC_FP32) {
    if (d->tile != 0 || d->splits != 1) return "the fp32 engine has one kernel: tile 0, splits 1";
  } else {
    const int t = d->tile;
    const bool pair = t == 32 || t == 64 || t == 96 || t == 128 || t == 192 || t == 256;
    if (pair ? N % t != 0 : (t == -128 ? N % 128 != 0 : ((t == 0 || t == -64) ? N % 64 != 0 : true)))
      return "tile must be 0, 32, 64, 96, 128, 192, 256, -64 or -128 and divide N";
  }
  switch (d->epi) {
    case EPI_QKV:
      if (d->D < 32 || d->D % 32 != 0 || N % d->D != 0 || d->sec0 < 0 || d->sec0 + N / d->D > 3)
        return "QKV: D % 32 == 0 and the columns sec0 .. sec0 + N / D - 1 within q, k, v";
      if (d->rpb < 1 || d->t0 < 0 || d->t_stride < d->t0 + d->rpb) return "QKV: cache slots t0 .. t0 + rpb - 1 within t_stride";
      if ((d->sec0 == 0 && d->q == nullptr) || d->kdst == nullptr || d->vdst == nullptr) return "QKV: q, kdst, vdst";
      break;
    case EPI_RESID:
      if (d->x == nullptr) return "RESID: x";
      break;
    case EPI_GELU:
      if (d->out == nullptr) return "GELU: out";
      break;
    default:
      if (d->outf == nullptr || d->ldo < N || d->ldo % 4 != 0 || d->split_stride % 4 != 0) return "F32: outf, ldo >= N, ldo % 4 == 0";
  }
  return nullptr;
}

extern "C" int hq_debug_gemm_epi(int prec, const void* A, const void* W, int w_rows, int M, int N, int K,
                                 const hq_debug_epi* d, void* stream) {
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const char* bad = (A == nullptr || W == nullptr || d == nullptr) ? "null operand" : debug_epi_invalid(prec, w_rows, M, N, K, d);
  if (bad != nullptr) {
    set_err(nullptr, "hq_debug_gemm_epi: %s", bad);
    return HQ_ERR_INVALID;
  }
  hq_ctx tmp;   // launch bookkeeping, the pinned tile width and ring-stage depth
  tmp.dbg.force_bn = d->tile;
  tmp.dbg.gemm_ks1 = d->ks1 != 0;
  if (prec == HQ_PREC_FP32) {
    // as gemm_any: the weight rows start w_row_off rows in
    const float* A32 = static_cast<const float*>(A);
    const float* W32 = static_cast<const float*>(W) + static_cast<size_t>(d->w_row_off) * K;
    const EpiParams<float> ep = debug_epi_params<float>(d);
    switch (d->epi) {
      case EPI_QKV: gemm_f32<EPI_QKV>(&tmp, st, A32, W32, M, N, K, ep); break;
      case EPI_RESID: gemm_f32<EPI_RESID>(&tmp, st, A32, W32, M, N, K, ep); break;
      case EPI_GELU: gemm_f32<EPI_GELU>(&tmp, st, A32, W32, M, N, K, ep); break;
      default: gemm_f32<EPI_F32>(&tmp, st, A32, W32, M, N, K, ep);
    }
  } else {
    tmp.prec = prec;
    int dev = 0;
    HQ_CUDA(nullptr, cudaGetDevice(&dev));
    int rc = check_device(&tmp, dev);
    if (rc == HQ_OK) rc = get_encode_fn(&tmp, &tmp.encode);
    if (rc == HQ_OK) rc = set_gemm_attrs_for(&tmp);
    // A rows padded to the 128-row tile by a zero-filled staging copy, as hq_debug_gemm
    const int Mp = (M + 127) / 128 * 128;
    void* Ap = nullptr;
    if (rc == HQ_OK) {
      HQ_CUDA(nullptr, cudaMalloc(&Ap, static_cast<size_t>(Mp) * K * 2));
      cudaMemsetAsync(Ap, 0, static_cast<size_t>(Mp) * K * 2, st);
      cudaMemcpyAsync(Ap, A, static_cast<size_t>(M) * K * 2, cudaMemcpyDeviceToDevice, st);
    }
    CUtensorMap mA, mA3, mW;
    PairMaps mWp;
    if (rc == HQ_OK) rc = make_map(&tmp, &mA, Ap, Mp, K, 128);
    if (rc == HQ_OK && K >= 128) rc = make_map3(&tmp, &mA3, Ap, Mp, K, 128, 2);
    if (rc == HQ_OK) rc = make_map(&tmp, &mW, const_cast<void*>(W), w_rows, K, 64);
    if (rc == HQ_OK) rc = make_pair_maps(&tmp, &mWp, const_cast<void*>(W), w_rows, K);
    if (rc == HQ_OK) {
      const CUtensorMap* a3 = K >= 128 ? &mA3 : nullptr;
      const int off = d->w_row_off;
      with_act(prec, [&](auto tag) {
        using AT = decltype(tag);
        if constexpr (sizeof(AT) == 2) {
          const EpiParams<AT> ep = debug_epi_params<AT>(d);
          switch (d->epi) {
            case EPI_QKV: gemm_tc<EPI_QKV, AT>(&tmp, st, mA, a3, mW, mWp, off, M, N, K, ep); break;
            case EPI_RESID: gemm_tc<EPI_RESID, AT>(&tmp, st, mA, a3, mW, mWp, off, M, N, K, ep); break;
            case EPI_GELU: gemm_tc<EPI_GELU, AT>(&tmp, st, mA, a3, mW, mWp, off, M, N, K, ep); break;
            default: gemm_tc<EPI_F32, AT>(&tmp, st, mA, a3, mW, mWp, off, M, N, K, ep, d->splits);
          }
        }
      });
    }
    cudaError_t se = cudaStreamSynchronize(st);
    if (Ap) cudaFree(Ap);
    if (rc != HQ_OK) {
      g_last_error = tmp.err;
      return rc;
    }
    if (se != cudaSuccess) {
      set_err(nullptr, "hq_debug_gemm_epi: %s", cudaGetErrorString(se));
      return HQ_ERR_CUDA;
    }
  }
  cudaError_t e = tmp.launch_err;
  if (e == cudaSuccess) e = cudaStreamSynchronize(st);
  if (e != cudaSuccess) {
    set_err(nullptr, "hq_debug_gemm_epi: %s", cudaGetErrorString(e));
    return HQ_ERR_CUDA;
  }
  return HQ_OK;
}

extern "C" int hq_debug_layernorm(int prec_out, float* x, const float* gamma, const float* beta, const float* add, void* out,
                                  int rows, int D, int in_group, int in_mul, int in_off, int out_mul, const float* fold,
                                  int n_fold, size_t fold_stride, const float* fold_bias, void* stream) {
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const char* bad = nullptr;
  if (prec_out != HQ_PREC_BF16 && prec_out != HQ_PREC_F16 && prec_out != HQ_PREC_FP32) bad = "unknown precision";
  else if (!x || !gamma || !beta || !out) bad = "null x, gamma, beta or out";
  else if (rows < 1 || D < 4 || D % 4 != 0) bad = "rows >= 1 and D % 4 == 0";
  else if (in_group < 1 || in_mul < 0 || in_off < 0 || out_mul < 1) bad = "row map";
  else if (n_fold < 0 || n_fold > LN_MAXFOLD || (n_fold > 0) != (fold != nullptr) || fold_stride % 4 != 0)
    bad = "fold: n_fold 0..6 partial sums, given iff n_fold > 0";
  if (bad != nullptr) {
    set_err(nullptr, "hq_debug_layernorm: %s", bad);
    return HQ_ERR_INVALID;
  }
  hq_ctx tmp;   // launch bookkeeping + the row width
  tmp.D = D;
  Fold f;
  f.partial = fold; f.n = n_fold; f.stride = fold_stride; f.bias = fold_bias;
  with_act(prec_out, [&](auto tag) {
    using AT = decltype(tag);
    layernorm_rows<AT>(&tmp, st, "layernorm", x, gamma, beta, add, static_cast<AT*>(out), rows, in_group, in_mul, in_off, out_mul,
                       f);
  });
  cudaError_t e = tmp.launch_err;
  if (e == cudaSuccess) e = cudaStreamSynchronize(st);
  if (e != cudaSuccess) {
    set_err(nullptr, "hq_debug_layernorm: %s", cudaGetErrorString(e));
    return HQ_ERR_CUDA;
  }
  return HQ_OK;
}

extern "C" int hq_debug_philox(uint64_t seed, const uint32_t counter[4], uint32_t out[4]) {
  uint32_t o[4];
  philox4x32_10(static_cast<uint32_t>(seed), static_cast<uint32_t>(seed >> 32), counter[0], counter[1], counter[2],
                counter[3], o);
  for (int i = 0; i < 4; ++i) out[i] = o[i];
  return HQ_OK;
}

extern "C" int hq_debug_sample(const float* logits, int R, int V, float temperature, int top_k, float top_p,
                               uint64_t seed, uint64_t row_offset, int position, int slot, int64_t* out_codes,
                               float* out_probs, void* stream) {
  if (!logits || !out_codes || R < 1 || V < 4 || V % 4 != 0 || V > 32768 || !(temperature > 0.f)) {
    set_err(nullptr, "hq_debug_sample: bad argument");
    return HQ_ERR_INVALID;
  }
  hq_ctx tmp;
  SampleArgs sa;
  memset(&sa, 0, sizeof(sa));
  sa.logits = logits; sa.ldl = V; sa.V = V; sa.R = R; sa.rows_per_b = 1; sa.slot0 = slot; sa.sp = nullptr;
  sa.pos = position; sa.S = 1; sa.flat_out = out_codes; sa.probs_out = out_probs; sa.Vmax = V; sa.n_slots = 5; sa.dst_w = 1;
  sa.temperature = temperature; sa.top_p = top_p; sa.top_k = top_k; sa.seed = seed; sa.row_offset = row_offset;
  sa.bot_slot = -1;
  launch_sample(&tmp, static_cast<cudaStream_t>(stream), sa);
  if (tmp.launch_err != cudaSuccess) {
    set_err(nullptr, "hq_debug_sample launch failed: %s", cudaGetErrorString(tmp.launch_err));
    return HQ_ERR_CUDA;
  }
  return HQ_OK;
}

extern "C" int hq_bench_attention(hq_ctx* ctx, int B, int n_keys, int iters, float* usec, void* stream) {
  if (!ctx || !usec || B < 1 || B > ctx->max_batch || n_keys < 1 || n_keys > ctx->Tc || iters < 1) {
    set_err(ctx, "hq_bench_attention: bad argument");
    return HQ_ERR_INVALID;
  }
  HQ_CUDA(ctx, cudaSetDevice(ctx->device));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  cudaEvent_t e0, e1;
  HQ_CUDA(ctx, cudaEventCreate(&e0));
  HQ_CUDA(ctx, cudaEventCreate(&e1));
  const size_t lstride = static_cast<size_t>(ctx->max_batch) * ctx->Tc * ctx->D;
  ctx->launch_err = cudaSuccess;
  struct PdlOff { hq_ctx* c; bool saved; PdlOff(hq_ctx* x) : c(x), saved(x->use_pdl) { x->use_pdl = false; } ~PdlOff() { c->use_pdl = saved; } } pdl_off(ctx);
  auto launch = [&](int l) {
    with_act(ctx->prec, [&](auto tag) {
      using AT = decltype(tag);
      AT* kc = static_cast<AT*>(ctx->kc) + l * lstride;
      AT* vc = static_cast<AT*>(ctx->vc) + l * lstride;
      attention<AT>(ctx, st, static_cast<AT*>(ctx->q), kc, vc, static_cast<AT*>(ctx->att.ptr), B, 1, ctx->Tc, n_keys, 0);
    });
  };
  for (int i = 0; i < 3; ++i) launch(i % ctx->L);
  HQ_CUDA(ctx, cudaEventRecord(e0, st));
  for (int i = 0; i < iters; ++i) launch(i % ctx->L);   // cycling layers: every launch reads a different cache slab
  HQ_CUDA(ctx, cudaEventRecord(e1, st));
  HQ_CUDA(ctx, cudaEventSynchronize(e1));
  float ms = 0.f;
  HQ_CUDA(ctx, cudaEventElapsedTime(&ms, e0, e1));
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  if (ctx->launch_err != cudaSuccess) {
    set_err(ctx, "attention launch failed: %s", cudaGetErrorString(ctx->launch_err));
    return HQ_ERR_CUDA;
  }
  *usec = ms * 1000.f / iters;
  return HQ_OK;
}

// One instrumented launch of the decode attention (after `warm` plain ones on other layers' slabs): per-CTA %globaltimer
// stamps at 8 points of the CTA's life (see phase_mark in kernels.cuh).  out_ns: [max_ctas][8], 0 = phase not reached.
extern "C" int hq_debug_attention_phases(hq_ctx* ctx, int B, int n_keys, int warm, unsigned long long* out_ns, int max_ctas,
                                         int* n_ctas, void* stream) {
  if (!ctx || !out_ns || !n_ctas || B < 1 || B > ctx->max_batch || n_keys < 1 || n_keys > ctx->Tc || max_ctas < 1) {
    set_err(ctx, "hq_debug_attention_phases: bad argument");
    return HQ_ERR_INVALID;
  }
  HQ_CUDA(ctx, cudaSetDevice(ctx->device));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  unsigned long long* dev = nullptr;
  const size_t bytes = static_cast<size_t>(max_ctas) * 8 * sizeof(unsigned long long);
  HQ_CUDA(ctx, cudaMalloc(reinterpret_cast<void**>(&dev), bytes));
  HQ_CUDA(ctx, cudaMemsetAsync(dev, 0, bytes, st));
  const size_t lstride = static_cast<size_t>(ctx->max_batch) * ctx->Tc * ctx->D;
  ctx->launch_err = cudaSuccess;
  struct PdlOff { hq_ctx* c; bool saved; PdlOff(hq_ctx* x) : c(x), saved(x->use_pdl) { x->use_pdl = false; } ~PdlOff() { c->use_pdl = saved; } } pdl_off(ctx);
  const int64_t before = ctx->launches;
  auto launch = [&](int l) {
    with_act(ctx->prec, [&](auto tag) {
      using AT = decltype(tag);
      AT* kc = static_cast<AT*>(ctx->kc) + l * lstride;
      AT* vc = static_cast<AT*>(ctx->vc) + l * lstride;
      attention<AT>(ctx, st, static_cast<AT*>(ctx->q), kc, vc, static_cast<AT*>(ctx->att.ptr), B, 1, ctx->Tc, n_keys, 0);
    });
  };
  for (int i = 0; i < warm; ++i) launch(i % ctx->L);
  HQ_CUDA(ctx, cudaStreamSynchronize(st));
  HQ_CUDA(ctx, cudaMemcpyToSymbol(g_hq_phase, &dev, sizeof(dev)));
  launch(warm % ctx->L);
  cudaError_t e = cudaStreamSynchronize(st);
  unsigned long long* null_ptr = nullptr;
  cudaMemcpyToSymbol(g_hq_phase, &null_ptr, sizeof(null_ptr));
  (void)before;
  if (e == cudaSuccess) e = ctx->launch_err;
  if (e == cudaSuccess) e = cudaMemcpy(out_ns, dev, bytes, cudaMemcpyDeviceToHost);
  cudaFree(dev);
  if (e != cudaSuccess) {
    set_err(ctx, "hq_debug_attention_phases: %s", cudaGetErrorString(e));
    return HQ_ERR_CUDA;
  }
  int n = 0;
  for (int i = 0; i < max_ctas; ++i)
    if (out_ns[static_cast<size_t>(i) * 8] != 0) n = i + 1;
  *n_ctas = n;
  return HQ_OK;
}

// Times one GEMM family of the sampler in isolation (events on `stream`): kind 0 = qkv [3D, D], 1 = proj [D, D],
// 2 = fc1 [4D, D], 3 = fc2 [D, 4D], 4 = head_top [V, D].  Successive launches cycle through the layers and a
// 256 MB scratch write between launches evicts L2, so every launch streams its weights from HBM as in the real loop.
extern "C" int hq_bench_gemm(hq_ctx* ctx, int kind, int M, int iters, float* usec, void* stream) {
  if (!ctx || !usec || kind < 0 || kind > 4 || M < 1 || M > ctx->h.rows || iters < 1) {
    set_err(ctx, "hq_bench_gemm: bad argument");
    return HQ_ERR_INVALID;
  }
  HQ_CUDA(ctx, cudaSetDevice(ctx->device));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int D = ctx->D;
  const size_t flush_bytes = static_cast<size_t>(256) << 20;
  void* flush = nullptr;
  HQ_CUDA(ctx, cudaMalloc(&flush, flush_bytes));
  std::vector<cudaEvent_t> ev(2 * iters);
  for (auto& e : ev) cudaEventCreate(&e);
  ctx->launch_err = cudaSuccess;
  struct PdlOff { hq_ctx* c; bool saved; PdlOff(hq_ctx* x) : c(x), saved(x->use_pdl) { x->use_pdl = false; } ~PdlOff() { c->use_pdl = saved; } } pdl_off(ctx);
  auto launch = [&](int i) {
    const BlockW& w = ctx->blocks[i % ctx->L];
    with_act(ctx->prec, [&](auto tag) {
      using AT = decltype(tag);
      EpiParams<AT> e;
      memset(&e, 0, sizeof(e));
      if (kind == 0) {
        e.bias = w.bqkv; e.q = static_cast<AT*>(ctx->q); e.kdst = static_cast<AT*>(ctx->kd); e.vdst = static_cast<AT*>(ctx->vd);
        e.D = D; e.rpb = 4; e.t_stride = 5; e.t0 = 1;
        gemm_any<EPI_QKV>(ctx, st, ctx->h, w.qkv, 0, M, 3 * D, D, e);
      } else if (kind == 1) {
        e.bias = w.bproj; e.x = ctx->yd;
        gemm_any<EPI_RESID>(ctx, st, ctx->att, w.proj, 0, M, D, D, e);
      } else if (kind == 2) {
        e.bias = w.b1; e.out = static_cast<AT*>(ctx->mlp.ptr);
        gemm_any<EPI_GELU>(ctx, st, ctx->h, w.fc1, 0, M, 4 * D, D, e);
      } else if (kind == 3) {
        e.bias = w.b2; e.x = ctx->yd;
        gemm_any<EPI_RESID>(ctx, st, ctx->mlp, w.fc2, 0, M, D, 4 * D, e);
      } else {
        e.outf = ctx->logits; e.ldo = ctx->Vmax;
        gemm_any<EPI_F32>(ctx, st, ctx->h, ctx->head_top, 0, M, ctx->Vt, D, e);
      }
    });
  };
  // rows >= max_batch of kd/vd would be out of range for the qkv epilogue: clamp M for kind 0
  if (kind == 0 && M > 4 * ctx->max_batch) M = 4 * ctx->max_batch;
  for (int i = 0; i < 3; ++i) launch(i);
  for (int i = 0; i < iters; ++i) {
    cudaMemsetAsync(flush, i & 0xff, flush_bytes, st);
    cudaEventRecord(ev[2 * i], st);
    launch(i);
    cudaEventRecord(ev[2 * i + 1], st);
  }
  cudaError_t se = cudaStreamSynchronize(st);
  double tot = 0.0;
  for (int i = 0; i < iters; ++i) {
    float ms = 0.f;
    cudaEventElapsedTime(&ms, ev[2 * i], ev[2 * i + 1]);
    tot += ms;
  }
  for (auto& e : ev) cudaEventDestroy(e);
  cudaFree(flush);
  if (se != cudaSuccess || ctx->launch_err != cudaSuccess) {
    set_err(ctx, "hq_bench_gemm: %s / %s", cudaGetErrorString(se), cudaGetErrorString(ctx->launch_err));
    return HQ_ERR_CUDA;
  }
  *usec = static_cast<float>(tot * 1000.0 / iters);
  return HQ_OK;
}

// ------------------------------------------------------------------------------------------------
// Stand-alone GEMM timing on synthetic operands (own allocations): per-launch CUDA-event times of the bf16 kernels
// for an arbitrary shape / tile.  flush: 0 = none (the W copies are cycled: `copies` distinct weight buffers),
// 1 = 256 MB memset before every launch (leaves L2 full of dirty lines), 2 = 256 MB read sweep (clean eviction).
// ------------------------------------------------------------------------------------------------
__global__ void read_sweep_kernel(const uint4* __restrict__ p, size_t n, unsigned* sink) {
  unsigned acc = 0;
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < n;
       i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const uint4 v = p[i];
    acc ^= v.x ^ v.y ^ v.z ^ v.w;
  }
  if (acc == 0x12345678u) *sink = acc;
}

extern "C" int hq_bench_gemm_shape(int M, int N, int K, int tile, int iters, int flush, int copies, float* usec_mean,
                                   float* usec_min, void* stream) {
  if (M < 1 || N % 64 != 0 || K % 64 != 0 || iters < 1 || copies < 1 || !usec_mean || !usec_min) {
    set_err(nullptr, "hq_bench_gemm_shape: bad argument");
    return HQ_ERR_INVALID;
  }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  hq_ctx tmp;
  const int splits = tmp.dbg.bench_splits > 0 ? tmp.dbg.bench_splits : 1;
  int dev = 0;
  HQ_CUDA(nullptr, cudaGetDevice(&dev));
  int rc = check_device(&tmp, dev);
  if (rc == HQ_OK) rc = get_encode_fn(&tmp, &tmp.encode);
  if (rc == HQ_OK) rc = set_gemm_attrs<bf16>(&tmp);
  if (rc != HQ_OK) {
    g_last_error = tmp.err;
    return rc;
  }
  const int Mp = (M + 127) / 128 * 128;
  void *A = nullptr, *W = nullptr, *flushbuf = nullptr;
  float* C = nullptr;
  unsigned* sink = nullptr;
  const size_t wbytes = static_cast<size_t>(N) * K * 2;
  const size_t flush_bytes = static_cast<size_t>(256) << 20;
  HQ_CUDA(nullptr, cudaMalloc(&A, static_cast<size_t>(Mp) * K * 2));
  HQ_CUDA(nullptr, cudaMalloc(&W, wbytes * copies));
  HQ_CUDA(nullptr, cudaMalloc(reinterpret_cast<void**>(&C), static_cast<size_t>(M) * N * 4 * splits));
  HQ_CUDA(nullptr, cudaMalloc(&flushbuf, flush_bytes));
  HQ_CUDA(nullptr, cudaMalloc(reinterpret_cast<void**>(&sink), 4));
  cudaMemsetAsync(A, 0, static_cast<size_t>(Mp) * K * 2, st);
  cudaMemsetAsync(W, 0, wbytes * copies, st);
  cudaMemsetAsync(flushbuf, 1, flush_bytes, st);
  long long* prof_buf = nullptr;
  CUtensorMap mA, mA3;
  std::vector<CUtensorMap> mW(copies);
  std::vector<PairMaps> mWp(copies);
  rc = make_map(&tmp, &mA, A, Mp, K, 128);
  if (rc == HQ_OK && K >= 128) rc = make_map3(&tmp, &mA3, A, Mp, K, 128, 2);
  for (int c = 0; rc == HQ_OK && c < copies; ++c) {
    rc = make_map(&tmp, &mW[c], static_cast<char*>(W) + wbytes * c, N, K, 64);
    if (rc == HQ_OK) rc = make_pair_maps(&tmp, &mWp[c], static_cast<char*>(W) + wbytes * c, N, K);
  }
  std::vector<cudaEvent_t> ev(2 * iters);
  for (auto& e : ev) cudaEventCreate(&e);
  if (rc == HQ_OK) {
    EpiParams<bf16> e;
    memset(&e, 0, sizeof(e));
    e.outf = C; e.ldo = N; e.split_stride = static_cast<size_t>(M) * N;
    if (getenv("HQ_GEMM_PROF") != nullptr && cudaMalloc(reinterpret_cast<void**>(&e.prof), 16 * sizeof(long long)) == cudaSuccess)
      cudaMemsetAsync(e.prof, 0, 16 * sizeof(long long), st);
    prof_buf = e.prof;
    tmp.dbg.force_bn = tile;
    for (int i = -3; i < iters; ++i) {
      const int c = ((i % copies) + copies) % copies;
      if (flush == 1) cudaMemsetAsync(flushbuf, i & 0xff, flush_bytes, st);
      if (flush == 2) read_sweep_kernel<<<1184, 256, 0, st>>>(static_cast<const uint4*>(flushbuf), flush_bytes / 16, sink);
      if (i >= 0) cudaEventRecord(ev[2 * i], st);
      gemm_tc<EPI_F32, bf16>(&tmp, st, mA, K >= 128 ? &mA3 : nullptr, mW[c], mWp[c], 0, M, N, K, e, splits);
      if (i >= 0) cudaEventRecord(ev[2 * i + 1], st);
    }
  }
  cudaError_t se = cudaStreamSynchronize(st);
  if (prof_buf != nullptr) {
    long long h[16];
    if (cudaMemcpy(h, prof_buf, sizeof(h), cudaMemcpyDeviceToHost) == cudaSuccess && h[8] > 0) {
      const double np = h[3] > 0 ? static_cast<double>(h[3]) : 1.0, nm = static_cast<double>(h[8]);
      fprintf(stderr,
              "[gemm prof] M=%d N=%d K=%d tile=%d (pair 0 leader, last launch; clk per ring stage) producer: wait_empty %.0f issue %.0f "
              "loop %.0f (n=%lld) | mma: wait_full %.0f issue %.0f commit %.0f loop %.0f (n=%lld)\n",
              M, N, K, tile, h[0] / np, h[1] / np, h[2] / np, h[3], h[4] / nm, h[5] / nm, h[6] / nm, h[7] / nm, h[8]);
    }
    cudaFree(prof_buf);
  }
  double tot = 0.0, mn = 1e30;
  for (int i = 0; i < iters; ++i) {
    float ms = 0.f;
    cudaEventElapsedTime(&ms, ev[2 * i], ev[2 * i + 1]);
    tot += ms;
    if (ms < mn) mn = ms;
  }
  for (auto& e : ev) cudaEventDestroy(e);
  cudaFree(A); cudaFree(W); cudaFree(C); cudaFree(flushbuf); cudaFree(sink);
  if (rc != HQ_OK) {
    g_last_error = tmp.err;
    return rc;
  }
  if (se != cudaSuccess || tmp.launch_err != cudaSuccess) {
    set_err(nullptr, "hq_bench_gemm_shape: %s / %s", cudaGetErrorString(se), cudaGetErrorString(tmp.launch_err));
    return HQ_ERR_CUDA;
  }
  *usec_mean = static_cast<float>(tot * 1000.0 / iters);
  *usec_min = static_cast<float>(mn * 1000.0);
  return HQ_OK;
}

// One hq_run as plain stream launches in which op `op_idx` of the `launch_idx`-th chain launch stamps %globaltimer per CTA:
// out_ns[8*c + p], p = 0 op begins, 1 grid barrier seen, 2 epilogue warps released, 3 work done, 4 proxy fence done,
// 5 all epilogue warps done, 6 arrival posted.  The op's tag (e.g. "layernorm", "gemm_qkv:...") is returned in `tag`.
extern "C" int hq_debug_chain_phases(hq_ctx* ctx, const hq_run_args* args, void* stream, int launch_idx, int op_idx,
                                     unsigned long long* out_ns, int max_ctas, int* n_ctas) {
  if (!ctx || !args || !out_ns || !n_ctas || max_ctas < 1 || launch_idx < 0 || op_idx < 0) return HQ_ERR_INVALID;
  HQ_CUDA(ctx, cudaSetDevice(ctx->device));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  unsigned long long* dev = nullptr;
  const size_t bytes = static_cast<size_t>(max_ctas) * 8 * sizeof(unsigned long long);
  HQ_CUDA(ctx, cudaMalloc(reinterpret_cast<void**>(&dev), bytes));
  HQ_CUDA(ctx, cudaMemset(dev, 0, bytes));
  HQ_CUDA(ctx, cudaMemcpyToSymbol(g_hq_chain_phase, &dev, sizeof(dev)));
  const int saved_graph = ctx->cfg.use_cuda_graph;
  ctx->cfg.use_cuda_graph = 0;
  ctx->phase_launch = launch_idx;
  ctx->phase_op = op_idx;
  int rc = run_impl(ctx, args, st, cudaMemcpyDeviceToDevice, cudaMemcpyDeviceToDevice);
  ctx->phase_launch = ctx->phase_op = -1;
  ctx->cfg.use_cuda_graph = saved_graph;
  cudaError_t e = cudaStreamSynchronize(st);
  unsigned long long* null_ptr = nullptr;
  cudaMemcpyToSymbol(g_hq_chain_phase, &null_ptr, sizeof(null_ptr));
  if (rc == HQ_OK && e == cudaSuccess) e = cudaMemcpy(out_ns, dev, bytes, cudaMemcpyDeviceToHost);
  cudaFree(dev);
  if (rc != HQ_OK) return rc;
  if (e != cudaSuccess) {
    set_err(ctx, "hq_debug_chain_phases: %s", cudaGetErrorString(e));
    return HQ_ERR_CUDA;
  }
  int n = 0;
  for (int i = 0; i < max_ctas; ++i)
    if (out_ns[static_cast<size_t>(i) * 8] != 0) n = i + 1;
  *n_ctas = n;
  return HQ_OK;
}

// ------------------------------------------------------------------------------------------------
// hq_trace_run: one hq_run with the per-kernel timeline recorded on the device (%globaltimer, ns).
// out_ns[2*i], out_ns[2*i+1] = first-CTA start / last-CTA end of launch i (in launch order); tags[i*24..] = kernel tag.
// ------------------------------------------------------------------------------------------------
extern "C" int hq_trace_run(hq_ctx* ctx, const hq_run_args* args, void* stream, unsigned long long* out_ns, char* tags,
                            int max_entries, int* n_entries) {
  if (!ctx || !args || !out_ns || !tags || !n_entries || max_entries < 1) return HQ_ERR_INVALID;
  HQ_CUDA(ctx, cudaSetDevice(ctx->device));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  unsigned long long* dbuf = nullptr;
  HQ_CUDA(ctx, cudaMalloc(reinterpret_cast<void**>(&dbuf), sizeof(unsigned long long) * 2 * max_entries));
  std::vector<unsigned long long> init(2 * static_cast<size_t>(max_entries));
  for (int i = 0; i < max_entries; ++i) { init[2 * i] = ~0ull; init[2 * i + 1] = 0ull; }
  HQ_CUDA(ctx, cudaMemcpy(dbuf, init.data(), init.size() * 8, cudaMemcpyHostToDevice));
  HQ_CUDA(ctx, cudaMemcpyToSymbol(g_hq_trace, &dbuf, sizeof(dbuf)));
  // drop a previously captured traced graph of this shape: its launch ids are baked in, the tags vector is rebuilt now
  for (auto it = ctx->graphs.begin(); it != ctx->graphs.end();) {
    if (it->first.tracing) { cudaGraphExecDestroy(it->second.exec); it = ctx->graphs.erase(it); } else ++it;
  }
  const bool saved_pdl = ctx->use_pdl;
  // with PDL a kernel is resident (waiting) long before it can run, so lifetimes overlap: off unless asked for
  if (!ctx->dbg.trace_pdl) ctx->use_pdl = false;
  ctx->tracing = true;
  ctx->trace_cap = max_entries;
  ctx->trace_tags.clear();
  ctx->trace_chain_cont.clear();
  int rc = run_impl(ctx, args, st, cudaMemcpyDeviceToDevice, cudaMemcpyDeviceToDevice);
  ctx->tracing = false;
  ctx->use_pdl = saved_pdl;
  cudaError_t se = cudaStreamSynchronize(st);
  if (rc == HQ_OK && se != cudaSuccess) {
    set_err(ctx, "hq_trace_run: %s", cudaGetErrorString(se));
    rc = HQ_ERR_CUDA;
  }
  if (rc == HQ_OK) {
    const int n = static_cast<int>(ctx->trace_tags.size());
    cudaMemcpy(out_ns, dbuf, sizeof(unsigned long long) * 2 * n, cudaMemcpyDeviceToHost);
    // ops of a chain launch: op i's span runs from the completion of op i-1 (grid barrier included) to its own
    ctx->trace_chain_cont.resize(static_cast<size_t>(n), 0);
    for (int i = 1; i < n; ++i)
      if (ctx->trace_chain_cont[i]) out_ns[2 * i] = out_ns[2 * (i - 1) + 1];
    for (int i = 0; i < n; ++i) {
      strncpy(tags + static_cast<size_t>(i) * 48, ctx->trace_tags[i].c_str(), 47);
      tags[static_cast<size_t>(i) * 48 + 47] = 0;
    }
    *n_entries = n;
  }
  unsigned long long* nullp = nullptr;
  cudaMemcpyToSymbol(g_hq_trace, &nullp, sizeof(nullp));
  cudaFree(dbuf);
  return rc;
}

// hq_debug_gemm_phases: hq_trace_run in which ONE launch (trace id `launch_id`, a CTA-pair GEMM) also stamps its per-CTA
// phases (gemm_tc2_kernel: 0 start, 1 prologue done, 2 dependency resolved, 3 first stage landed, 4 last MMA issued,
// 5 accumulator complete, 6 epilogue done, 7 end); phases[cta * 8 + p] in ns of %globaltimer, 0 = not stamped.
extern "C" int hq_debug_gemm_phases(hq_ctx* ctx, const hq_run_args* args, void* stream, int launch_id,
                                    unsigned long long* phases, int max_ctas, unsigned long long* out_ns, char* tags,
                                    int max_entries, int* n_entries) {
  if (!ctx || !phases || max_ctas < 1 || launch_id < 0) return HQ_ERR_INVALID;
  HQ_CUDA(ctx, cudaSetDevice(ctx->device));
  unsigned long long* dev = nullptr;
  const size_t bytes = static_cast<size_t>(max_ctas) * 16 * sizeof(unsigned long long);
  HQ_CUDA(ctx, cudaMalloc(reinterpret_cast<void**>(&dev), bytes));
  HQ_CUDA(ctx, cudaMemset(dev, 0, bytes));
  HQ_CUDA(ctx, cudaMemcpyToSymbol(g_hq_gemm_phase, &dev, sizeof(dev)));
  HQ_CUDA(ctx, cudaMemcpyToSymbol(g_hq_phase_id, &launch_id, sizeof(launch_id)));
  int rc = hq_trace_run(ctx, args, stream, out_ns, tags, max_entries, n_entries);
  unsigned long long* null_ptr = nullptr;
  const int none = -1;
  cudaMemcpyToSymbol(g_hq_gemm_phase, &null_ptr, sizeof(null_ptr));
  cudaMemcpyToSymbol(g_hq_phase_id, &none, sizeof(none));
  cudaError_t e = cudaSuccess;
  if (rc == HQ_OK) e = cudaMemcpy(phases, dev, bytes, cudaMemcpyDeviceToHost);
  cudaFree(dev);
  if (rc != HQ_OK) return rc;
  if (e != cudaSuccess) {
    set_err(ctx, "hq_debug_gemm_phases: %s", cudaGetErrorString(e));
    return HQ_ERR_CUDA;
  }
  return HQ_OK;
}

#include "stage1_host.cuh"
