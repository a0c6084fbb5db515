/*
 * hqgraft.h - C ABI of libhqgraft.so: the B200 (sm_100a) engine behind HQ-Transformer's
 * locally hierarchical autoregressive sampling loop.
 *
 * The reference (kakaobrain/hqtransformer) is pure Python and has no FFI; the boundary it exposes
 * for this path is Python-level (SURVEY.md section 8b).  Each entry point below states which
 * reference interface it stands behind (paths relative to the reference root).  The Python host
 * (hqtransformer_b200/) binds these with ctypes and re-exposes the reference's own call
 * signatures; INTEGRATION.md shows the stub a reference maintainer would add.
 *
 * Conventions
 *   - every function returns an int status (HQ_OK == 0); nothing throws across the boundary;
 *     hq_last_error() gives the message of the last failure (per ctx, or global when ctx==NULL);
 *   - plain pointers and sizes only; all tensors are caller-owned; device pointers must stay valid
 *     until the work enqueued on `stream` has completed; hq_run is asynchronous on `stream`;
 *   - a ctx belongs to one GPU and is not thread-safe;
 *   - sm_100a only, no CPU fallback: hq_create fails on any other device.
 */
#ifndef HQGRAFT_H_
#define HQGRAFT_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define HQ_ABI_VERSION 9

enum hq_status {
  HQ_OK = 0,
  HQ_ERR_INVALID = 1,      /* bad argument / shape / name */
  HQ_ERR_CUDA = 2,         /* CUDA runtime or driver error */
  HQ_ERR_UNSUPPORTED = 3,  /* device is not sm_100, or config outside the supported envelope */
  HQ_ERR_STATE = 4         /* call order (e.g. hq_run before every parameter was loaded) */
};

enum hq_cond_kind { HQ_COND_CLS = 0, HQ_COND_TXT = 1, HQ_COND_UNCOND = 2 };

/* HQ_PREC_BF16: bf16 weights / GEMM inputs / KV cache, fp32 accumulate, residual, LayerNorm, softmax
 *               (tcgen05 + TMA GEMMs) - the engine `use_fp16=True` selects by default, the same split as the
 *               reference's fp16 autocast (torch.cuda.amp.autocast, hierarchical_ar.py:445) with bf16 for fp16.
 * HQ_PREC_FP32: everything fp32 on CUDA cores - the reference's `use_fp16=False`; used for the
 *               bit-exact greedy parity tests.
 * HQ_PREC_F16:  the bf16 engine with IEEE fp16 as the 2-byte type - the reference's own autocast format.  Rounded to
 *               fp16: GEMM weights, GEMM-input activations (LayerNorm outputs, attention outputs, GELU outputs), q / k / v
 *               and the KV cache.  fp32: accumulation, biases, the residual stream, LayerNorm statistics, softmax, logits
 *               and the sampler (the same kernels and rounding points as HQ_PREC_BF16).  No saturation or overflow
 *               detection: an activation beyond the fp16 range (|x| > 65504) becomes inf, as under the reference's
 *               autocast.  use_chain is ignored (no persistent chain kernel); fuse_head_sampler applies.  Libraries
 *               older than this value reject it in hq_create (HQ_ERR_INVALID).
 * HQ_PREC_TF32: stage-1 decoder only (hq_s1_config.precision; hq_create rejects it with HQ_ERR_INVALID) - what the
 *               reference's decode_code computes (fp32 outside autocast, cuDNN convolutions in TF32).  Convolutions on
 *               tcgen05 kind::tf32 with fp32 accumulation.  Rounded to TF32 (round-to-nearest, ties away from zero; stored
 *               as fp32 with the low 13 bits zero): every convolution input - codebook gather + PixelShuffle, GroupNorm(+swish)
 *               outputs, the copies of x that feed nin_shortcut and the upsample convolutions, attention outputs - and the
 *               conv weights.  fp32: q / k / v (unrounded), the AttnBlock core (CUDA cores), the residual stream, GroupNorm
 *               statistics, biases and the output image.  fp32 range throughout (no overflow at fp16's 65504). */
enum hq_precision { HQ_PREC_BF16 = 0, HQ_PREC_FP32 = 1, HQ_PREC_F16 = 2, HQ_PREC_TF32 = 3 };

enum hq_dtype { HQ_F32 = 0, HQ_BF16 = 1, HQ_F16 = 2 };

/* Depth-transformer schedule = the reference's `model_type` (hqvae/models/__init__.py:123-137):
 *   HQ_MODEL_PARALLEL       'parallel'       top, then the four bottoms in one pass (hierarchical_ar.py:667-789)
 *   HQ_MODEL_TOP2BOT        'top2bot'        five sequential single-token passes with a causal depth cache (:565-664)
 *   HQ_MODEL_BIDIRECTIONAL  'bidirectional'  one pass over [hs + sos_depth, pos_emb_depth[0..3]], unmasked (:791-878);
 *                                            as in the reference every token is drawn with the BOTTOM filters and
 *                                            softmax_temperature[0] */
enum hq_model_type { HQ_MODEL_PARALLEL = 0, HQ_MODEL_TOP2BOT = 1, HQ_MODEL_BIDIRECTIONAL = 2 };

/* Input embedding of the spatial transformer = hparams.embedding_type (hierarchical_ar.py:83-113, 516-548):
 *   HQ_EMB_TRANSFORMER1  mean over the five stack tokens of (embedding + pos_emb_emb) - ImageNet / CC-15M checkpoints
 *   HQ_EMB_REDUCE        tok_emb_top + the four D/4-wide bottom embeddings interleaved ('B (U L) K -> B U (K L)') - FFHQ */
enum hq_embedding_kind { HQ_EMB_TRANSFORMER1 = 0, HQ_EMB_REDUCE = 1 };

/* hparams.position_embedding (hierarchical_ar.py:118-125, 506-514): one table, or pos_emb_top_h[p / H] + pos_emb_top_w[p % H]
 * with H = sqrt(ctx_len_img) rows per table. */
enum hq_position_kind { HQ_POS_1D = 0, HQ_POS_2D = 1 };

/* Architecture of an iHQGPT (2-level HQ-Transformer; model_type / embedding_type / position_embedding variants below)
 * - constructor arguments at hqvae/models/stage2/hierarchical_ar.py:24-216, YAML fields at
 * hqvae/utils/config2.py:49-105. */
typedef struct hq_config {
  int32_t embed_dim;       /* hparams.embed_dim (multiple of 64; head size must be 64) */
  int32_t n_heads;         /* hparams.n_heads */
  int32_t n_layers;        /* hparams.n_layers (spatial transformer) */
  int32_t n_layers_depth;  /* hparams_dec.n_layers, 4 when hparams_dec is absent (:150-153) */
  int32_t vocab_top;       /* vocab_size_top */
  int32_t vocab_bot;       /* vocab_size_bot */
  int32_t vocab_txt;       /* vocab_size_txt (HQ_COND_TXT only) */
  int32_t n_classes;       /* hparams.n_classes (HQ_COND_CLS only) */
  int32_t ctx_len_img;     /* rows of pos_emb_top */
  int32_t ctx_len_txt;     /* text prefix length (HQ_COND_TXT only) */
  int32_t cond_kind;       /* hq_cond_kind */
  int32_t precision;       /* hq_precision */
  int32_t max_seq_len;     /* number of top positions a run may cover (64 for 8x8) */
  int32_t use_cuda_graph;  /* 1: capture each run shape once and replay it; 0: plain stream launches */
  int32_t use_pdl;         /* 1: chain the kernels with programmatic dependent launch (prologue of kernel n+1 and
                              its first weight tiles overlap the tail of kernel n); 0: plain stream order */
  int32_t use_chain;       /* 1 (bf16 engine only, batches > 128): the depth transformer of a position
                              (sampling_step_depth_parallel, hierarchical_ar.py:667-719) and the GEMM / LayerNorm runs of the
                              spatial blocks execute as persistent multi-op kernels (one launch per run of dependent ops,
                              grid barrier between ops); 0: one kernel per op.  Results are bit-identical either way. */
  int32_t model_type;      /* hq_model_type */
  int32_t embedding_kind;  /* hq_embedding_kind */
  int32_t position_kind;   /* hq_position_kind */
  int32_t code_levels;     /* 2: iHQGPT (1 top + 4 bottom codes per position); 3: the multi-level `HQTransformer`
                              (hqvae/models/stage2/hqtransformer.py, decoding_type 'parallel-add', embedding 'transformer1'):
                              1 top + 4 middle + 16 bottom codes per position in three depth passes.  0 is read as 2. */
  int32_t vocab_mid;       /* code_levels == 3: vocab_sizes[1] (vocab_top = vocab_sizes[0], vocab_bot = vocab_sizes[2]) */
  int32_t fuse_head_sampler; /* 1 (bf16 and fp16 engines): a draw with top_k None and top_p None (the measure_throughput protocol) is made
                              inside the head GEMM's epilogue - exact two-stage categorical sampling over 32-column chunks,
                              the [rows, V] logits are never written.  Same distribution as the unfused sampler, different
                              Philox counters (so a different, equally valid stream for a given seed); greedy, top-k, top-p,
                              teacher-forced and logits-returning runs always use the unfused sampler.  0: always unfused. */
} hq_config;

/* Arguments of Sample(z; T, k, p) - hierarchical_ar.py:762-785 with utils/sampling.py:12-37.
 * top_k <= 0 means None (no top-k cut); top_p <= 0 or >= 1 means no nucleus cut.
 * top_k == 1 is greedy: the lowest index among the maxima (the reference draws randomly among
 * exact ties; see DESIGN.md).
 * Every draw uses Philox4x32-10 keyed by `seed` with counter (row_offset + row, position, slot),
 * so results do not depend on how a batch is sharded over GPUs. */
typedef struct hq_sampling_params {
  int32_t top_k_top;
  int32_t top_k_bot;
  float top_p_top;
  float top_p_bot;
  float temperature_top;   /* softmax_temperature[0] */
  float temperature_bot;   /* softmax_temperature[1] */
  uint64_t seed;
  uint64_t row_offset;     /* global index of this shard's first row */
  int32_t top_k_mid;       /* middle level of the 3-level model: top_k[1], top_p[1], softmax_temperature[1] */
  float top_p_mid;         /* (hqtransformer.py:626-631); top = level 0, bot = level 2 there */
  float temperature_mid;
  int32_t reserved;
} hq_sampling_params;

/* One call of the sampling loop over top positions [pos_begin, pos_end).
 * Replaces the body of `sampling_ihqgpt` (hqvae/utils/sampling.py:164-237) and, with
 * pos_end == pos_begin + 1, one `iHQGPT.sampling_step` (hierarchical_ar.py:428-480).
 * pos_begin == 0 starts a new batch (resets the KV cache); pos_begin > 0 continues the batch whose
 * codes for positions < pos_begin are read from codes_top / codes_bot. */
typedef struct hq_run_args {
  int32_t batch;             /* B <= max_batch */
  int32_t seq_len;           /* S: row stride of the code / logits arrays (<= max_seq_len) */
  int32_t pos_begin;
  int32_t pos_end;
  const int64_t* cond;       /* [B] class ids | [B, ctx_len_txt] text ids | NULL (uncond) */
  const float* sos;          /* optional [B, T0, D] fp32 start embedding overriding `cond`
                                (T0 = ctx_len_txt for text, else 1) - the `sos` argument of
                                sampling_step (hierarchical_ar.py:430) */
  const int64_t* given_top;  /* optional [B, S]: forced top codes (given_top_code, sampling.py:205-208) */
  const int64_t* given_bot;  /* optional [B, S, 4]: forced bottom codes (teacher forcing, parity only) */
  int64_t* codes_top;        /* in/out [B, S] */
  int64_t* codes_bot;        /* in/out [B, S, 4], within-stack order j = kh*2 + kw  (code_levels == 3: [B, S, 16], raster
                                order of the 4x4 cell) */
  float* logits;             /* optional out [B, S, 5, max vocab] raw head outputs (code_levels == 3: [B, S, 21, max vocab]) */
  hq_sampling_params sampling;
  int64_t* codes_mid;        /* code_levels == 3 only: in/out [B, S, 4] middle codes, raster order of the 2x2 cell */
  const int64_t* given_mid;  /* code_levels == 3 only: optional forced middle codes (teacher forcing, parity only) */
  int32_t shared_prefix;     /* text models, pos_begin == 0: 1 = every row of `cond` is the SAME prompt (one prompt sampled B
                                times, as the reference notebook does): the 64-token prefill runs for row 0 only and its
                                cached keys / values are broadcast to the other rows.  Results are identical to 0.
                                With prefix_len > 0 (any model, `sos` NULL): 1 = every row has the same `cond` AND the same
                                prefix codes; the prefix pass runs for row 0 only and its cache rows are broadcast. */
  int32_t prefix_len;        /* image completion: 0 = off.  P in [1, pos_end) with pos_begin == 0: the codes of positions < P are
                                GIVEN - read from codes_top / codes_bot (/ codes_mid) and returned unchanged - and positions
                                [P, pos_end) are sampled exactly as the loop samples them after those codes (same Philox
                                counters).  The spatial KV cache of the prefix is computed in one causal pass over its
                                T0 + P - 1 tokens (no depth pass, head or draw there).  given_top / given_bot / given_mid apply
                                at positions >= P; logits are written for positions >= P only. */
} hq_run_args;

typedef struct hq_ctx hq_ctx;

int hq_abi_version(void);

/* Message of the last failure on `ctx` (or of the last failed hq_create when ctx == NULL). */
const char* hq_last_error(const hq_ctx* ctx);

/* Allocates the weight arena, the KV cache ([L][B][T][D] keys and values), workspaces and TMA
 * descriptors on `device` for batches of up to `max_batch` rows.
 * Stands behind `iHQGPT.__init__` (hierarchical_ar.py:24-216) followed by `.to('cuda')`
 * (sampling_hqmodel.py:80, measure_throughput/__main__.py:56). */
int hq_create(const hq_config* cfg, int device, int max_batch, hq_ctx** out);

int hq_destroy(hq_ctx* ctx);

/* Re-sizes the batch-dependent state (KV cache, activations, code buffers) for batches of up to
 * `max_batch` rows; parameters stay loaded.  The reference allocates this state implicitly on every
 * call (`past` list of tensors, sampling.py:227-231); here it is explicit and reused. */
int hq_reserve_batch(hq_ctx* ctx, int max_batch);
int hq_max_batch(const hq_ctx* ctx);

/* Copies one parameter into the engine layout (q/k/v fused to [3D, D]; GEMM weights cast to bf16 in
 * HQ_PREC_BF16 and to fp16 in HQ_PREC_F16, from fp32, bf16 or fp16 sources; everything else stays fp32).  `name` is the reference state_dict key without the 'stage2.' prefix, e.g.
 * "blocks.3.attn.query.weight", "depths.0.mlp.2.bias", "tok_emb_top.weight", "sos_depth", "head_bot.weight"
 * (module definitions hierarchical_ar.py:63-209, layers.py:43-52, 290-317).
 * Stands behind `load_state_dict(strict=True)` (sampling_hqmodel.py:79): unknown names and wrong
 * shapes are errors.  `data` may be a host (is_device == 0) or device pointer; the call is synchronous. */
int hq_load_param(hq_ctx* ctx, const char* name, const void* data, int dtype,
                  const int64_t* shape, int ndim, int is_device);

/* HQ_OK once every parameter the config requires has been loaded; otherwise HQ_ERR_STATE and
 * hq_last_error() lists the missing names (strict=True semantics). */
int hq_params_complete(hq_ctx* ctx);

/* The sampling loop.  All pointers in `args` are DEVICE pointers; asynchronous on `stream`
 * (a cudaStream_t; NULL = legacy default stream). */
int hq_run(hq_ctx* ctx, const hq_run_args* args, void* stream);

/* Same, but every pointer in `args` is a HOST pointer: inputs are copied host->device, the loop
 * runs, and the code grids (and logits, if requested) are copied back before the call returns.
 * This is the end-to-end call the reference scripts make (sampling_hqmodel.py:106-117 receives
 * host-visible code tensors it then rearranges and pickles). */
int hq_run_host(hq_ctx* ctx, const hq_run_args* args);

/* Number of kernel launches enqueued by the last hq_run / hq_run_host (graph nodes when replayed). */
int64_t hq_last_launch_count(const hq_ctx* ctx);

/* Launches of the persistent chain kernel (hq_config.use_chain) enqueued or captured since hq_create; 0 means every op
 * ran as a kernel of its own (batch <= 128, fp32 or fp16 engine, use_chain == 0). */
int64_t hq_chain_launch_count(const hq_ctx* ctx);

/* Bytes of device memory owned by the ctx (weights + KV cache + workspaces, including the image-completion workspace that
 * the first run with a longer prefix (or a larger batch under one) grows; hq_reserve_batch frees it). */
size_t hq_device_bytes(const hq_ctx* ctx);

/* ---- test / measurement hooks (used by tests/ and bench.py, not by the sampling entry points) ---- */

/* C[M,N] = A[M,K] * W[N,K]^T through the same tcgen05/TMA kernels the sampler uses (prec == HQ_PREC_BF16 / HQ_PREC_F16,
 * A and W bf16 / fp16) or the fp32 CUDA-core kernel (HQ_PREC_FP32, A and W fp32); C fp32; device pointers.
 * tile: 0 = the engine's own choice; 32/64/96/128/192/256 = CTA-pair kernel with that tile width;
 * -64 / -128 = single-CTA kernel. */
int hq_debug_gemm(int prec, const void* A, const void* W, float* C, int M, int N, int K, int tile, void* stream);

/* Fused epilogue of one hq_debug_gemm_epi launch (the sampler's EpiParams).  Device pointers; q, kdst, vdst, vdup and out
 * in the precision's activation type (bf16 | fp16 | fp32), bias, x and outf fp32. */
typedef struct hq_debug_epi {
  int32_t epi;          /* 0 QKV, 1 RESID, 2 GELU, 3 F32 (the sampler's EPI_* values) */
  int32_t tile;         /* as hq_debug_gemm's `tile` (bf16 / fp16; the fp32 engine has one kernel: 0) */
  int32_t ks1;          /* 1: one 64-wide k-block per ring stage even where the engine would stage two */
  int32_t D, sec0, rpb, t_stride, t0;   /* QKV: column n is section sec0 + n / D (0 q, 1 k, 2 v); row m goes to q[m] and
                                           to cache row (m / rpb) * t_stride + t0 + m % rpb of kdst / vdst */
  int32_t w_row_off;    /* the product uses W rows w_row_off .. w_row_off + N - 1 */
  int32_t ldo, splits;  /* F32: row stride of outf; K slices, slice s writes outf + s * split_stride (bf16 / fp16 only) */
  int32_t reserved;
  uint64_t split_stride;
  const float* bias;    /* [N] or NULL; QKV / RESID / GELU */
  void* q;              /* QKV: [M, D] (sec0 == 0) */
  void* kdst;
  void* vdst;
  void* vdup;           /* QKV: optional [M, D] second copy of the v columns */
  float* x;             /* RESID: [M, N], x += C + bias */
  void* out;            /* GELU: [M, N] = gelu(C + bias) */
  float* outf;          /* F32: [M, ldo] per K slice */
} hq_debug_epi;

/* C = A[M,K] * W[w_row_off .. w_row_off + N - 1, K]^T (W has w_rows rows) through the sampler's GEMM kernels and the
 * epilogue `e` describes, synchronously on `stream`.  HQ_ERR_INVALID for combinations the engine never launches
 * (a tile that does not divide N, splits that do not divide K / 64, split-K outside EPI_F32, ...). */
int hq_debug_gemm_epi(int prec, const void* A, const void* W, int w_rows, int M, int N, int K, const hq_debug_epi* e,
                      void* stream);

/* The sampler's LayerNorm launch: out[r * out_mul] = LN(x[(r / in_group) * in_mul + in_off + r % in_group]) * gamma + beta
 * (+ add), rows r < rows, out bf16 (prec_out == HQ_PREC_BF16), fp16 (HQ_PREC_F16) or fp32.  n_fold > 0: x row += fold_bias + the n_fold
 * partial sums fold + s * fold_stride (same row index), written back before the normalisation.  fp32 device pointers. */
int hq_debug_layernorm(int prec_out, float* x, const float* gamma, const float* beta, const float* add, void* out, int rows,
                       int D, int in_group, int in_mul, int in_off, int out_mul, const float* fold, int n_fold,
                       size_t fold_stride, const float* fold_bias, void* stream);

/* Philox4x32-10 block for (seed, counter) - known-answer test of the RNG; host pointers. */
int hq_debug_philox(uint64_t seed, const uint32_t counter[4], uint32_t out[4]);

/* Sample(z; T, k, p) on device logits [R, V] (fp32): writes int64 codes [R]; `slot` selects the
 * Philox counter lane, row r uses counter (row_offset + r, position, slot). */
int hq_debug_sample(const float* logits, int R, int V, float temperature, int top_k, float top_p,
                    uint64_t seed, uint64_t row_offset, int position, int slot,
                    int64_t* out_codes, float* out_probs /* optional [R, V] */, void* stream);

/* Single-query attention of B rows over `n_keys` cached keys through the kernels the sampler uses: q / out [B, D],
 * K / V [B, t_stride, D] with D = n_heads * 64, device pointers in the precision's activation type (bf16 / fp16 / fp32).
 * variant: 0 = the engine's choice (bf16 / fp16: persistent ldmatrix/mma kernel), 1 = the scalar bulk-staged kernel. */
int hq_debug_attention(int prec, const void* q, const void* K, const void* V, void* out, int B, int n_heads,
                       int t_stride, int n_keys, int variant, void* stream);

/* Causal attention of the image-completion prefix pass: query i of image b (q / out [B, n_q, D]) over keys 0 .. i of its
 * cache rows (K / V [B, t_stride, D]), D = n_heads * 64, device pointers in the precision's activation type.
 * variant 0: the kernel of the prefix pass - bf16 / fp16: the tensor-core prefix kernel, fp32: the per-(query, head) warp
 * kernel the fp32 engine runs there; variant 1: the per-(query, head) warp kernel at every precision (what the text prefill
 * runs).  1 <= n_q <= min(t_stride, 128). */
int hq_debug_attention_prefix(int prec, const void* q, const void* K, const void* V, void* out, int B, int n_heads,
                              int t_stride, int n_q, int variant, void* stream);

/* Times the single-query KV-cache attention kernel alone at cache length `n_keys` for batch B on the
 * ctx's cache (events on `stream`); returns mean microseconds over `iters` launches in *usec. */
int hq_bench_attention(hq_ctx* ctx, int B, int n_keys, int iters, float* usec, void* stream);

/* One instrumented launch of the decode attention at cache length `n_keys` after `warm` plain ones: out_ns[8*c + p] =
 * %globaltimer (ns) at which CTA c passed point p (0 start, 1 barriers ready, 2 q ready, 3 first keys landed, 4 scores
 * done, 5 softmax done, 6 first item written, 7 CTA end); *n_ctas = CTAs that reported. */
int hq_debug_attention_phases(hq_ctx* ctx, int B, int n_keys, int warm, unsigned long long* out_ns, int max_ctas,
                              int* n_ctas, void* stream);

/* One hq_run (device pointers, plain stream launches) in which op `op_idx` of the `launch_idx`-th persistent chain launch
 * stamps %globaltimer per CTA: out_ns[8*c + p], p = 0 op begins, 1 grid barrier seen, 2 epilogue warps released, 3 work done,
 * 4 proxy fence done, 5 all epilogue warps of the CTA done, 6 arrival posted; *n_ctas = CTAs that reported. */
int hq_debug_chain_phases(hq_ctx* ctx, const hq_run_args* args, void* stream, int launch_idx, int op_idx,
                          unsigned long long* out_ns, int max_ctas, int* n_ctas);

/* Times one GEMM family of the loop alone on the ctx's own weights and buffers: kind 0 = fused qkv [3D, D],
 * 1 = attention proj [D, D], 2 = mlp fc1 [4D, D], 3 = mlp fc2 [D, 4D], 4 = head_top [V, D]; M rows.  L2 is evicted
 * between launches (256 MB write) and layers are cycled, so weights stream from HBM as in the real loop. */
int hq_bench_gemm(hq_ctx* ctx, int kind, int M, int iters, float* usec, void* stream);

/* One hq_run (device pointers) with the kernel timeline recorded on the device: out_ns[2i] / out_ns[2i+1] = first-CTA
 * start / last-CTA end (%globaltimer, ns) of the i-th kernel launch, tags[48*i] = its NUL-terminated tag
 * (GEMMs carry their shape as ":MxNxK:s<splits>", the decode attention its cache length as ":t<keys>:B<rows>"). */
int hq_trace_run(hq_ctx* ctx, const hq_run_args* args, void* stream, unsigned long long* out_ns, char* tags,
                 int max_entries, int* n_entries);

/* hq_trace_run in which the launch with trace index `launch_id` (a CTA-pair GEMM) also stamps its per-CTA phases:
 * phases[16*c + p] = %globaltimer (ns) of CTA c at p = 0 start, 1 prologue done, 2 dependency resolved (griddepcontrol.wait
 * returned), 3 first ring stage landed, 4 last MMA issued, 5 accumulator complete, 6 epilogue done, 7 end, 8 / 9 / 10 first epilogue
 * chunk read from TMEM / parked in shared memory / stored; 0 = not stamped.  `phases` holds 16 * max_ctas values. */
int hq_debug_gemm_phases(hq_ctx* ctx, const hq_run_args* args, void* stream, int launch_id, unsigned long long* phases,
                         int max_ctas, unsigned long long* out_ns, char* tags, int max_entries, int* n_entries);

/* Stand-alone timing of the bf16 GEMM kernels on synthetic operands of any shape / tile (see hq_debug_gemm for
 * `tile`).  flush: 0 none (cycles `copies` weight buffers), 1 = 256 MB memset before each launch, 2 = 256 MB read
 * sweep before each launch.  Per-launch CUDA-event times; mean and min in microseconds. */
int hq_bench_gemm_shape(int M, int N, int K, int tile, int iters, int flush, int copies, float* usec_mean,
                        float* usec_min, void* stream);

/* ---- stage-1 decode of the sampled code grids (SURVEY.md 8f-1) ----
 * Stands behind `SimRQGAN2Generator.decode_code(code_t [B,h,w], code_b [B,2h,2w])` (hqvae/models/stage1/generator.py:323-367)
 * as the scripts call it after sampling (sampling_hqmodel.py:197, measure_throughput/__main__.py:108-111: one image at a
 * time there, batched here), for the shipped HQ-VAE configuration: `decoding_type: concat`, `upsample: pixelshuffle`,
 * `use_init_downsample / use_mid_block / use_attn: True` (the `stage1` section of the stage-2 YAMLs). */
typedef struct hq_s1_config {
  int32_t embed_dim;        /* stage1.embed_dim: bottom codebook width; the top codebook is 4x as wide (PixelShuffle(2)) */
  int32_t n_embed;          /* stage1.n_embed */
  int32_t z_channels;       /* hparams.z_channels */
  int32_t resolution;       /* hparams.resolution (pixels) */
  int32_t ch;               /* hparams.ch */
  int32_t ch_mult[8];       /* hparams.ch_mult[0 .. n_levels) */
  int32_t n_levels;         /* len(ch_mult); the bottom grid is resolution / 2^n_levels wide */
  int32_t num_res_blocks;   /* hparams.num_res_blocks */
  int32_t attn_resolution;  /* hparams.attn_resolutions[0] */
  int32_t out_ch;           /* hparams.out_ch (3) */
  int32_t precision;        /* HQ_PREC_BF16 (0, the default: bf16 convolution inputs and weights) or HQ_PREC_TF32 */
} hq_s1_config;

typedef struct hq_s1_ctx hq_s1_ctx;

int hq_s1_create(const hq_s1_config* cfg, int device, int max_batch, hq_s1_ctx** out);
int hq_s1_destroy(hq_s1_ctx* ctx);
const char* hq_s1_last_error(const hq_s1_ctx* ctx);
size_t hq_s1_device_bytes(const hq_s1_ctx* ctx);

/* `name`: key of the reference generator's state_dict without the 'stage1.' prefix, e.g. "quantize_t.embedding",
 * "post_quant_conv_b.weight", "decoder.up.2.block.1.conv1.weight", "decoder.mid.attn_1.q.bias" (generator.py:243-250,
 * stage1/modules/layers.py:77-186, 300-383).  Only the keys decode_code reads exist; conv weights (fp32, bf16 or fp16
 * sources) are repacked to [Cout, kh kw Cin] bf16, or fp32 rounded to TF32 under HQ_PREC_TF32.  hq_s1_params_complete: HQ_OK once all of them were loaded. */
int hq_s1_load_param(hq_s1_ctx* ctx, const char* name, const void* data, int dtype, const int64_t* shape, int ndim,
                     int is_device);
int hq_s1_params_complete(hq_s1_ctx* ctx);

/* code_t int64 [B, h, w], code_b int64 [B, 2h, 2w] -> out fp32 [B, out_ch, resolution, resolution]; DEVICE pointers,
 * asynchronous on `stream`; B <= max_batch.  Codes must lie in [0, n_embed) (the host layer checks). */
int hq_s1_decode_codes(hq_s1_ctx* ctx, const int64_t* code_t, const int64_t* code_b, float* out, int B, void* stream);

/* 2 * MACs of the convolutions of the last hq_s1_decode_codes call (interior pixels only): the roofline numerator. */
double hq_s1_last_conv_flops(const hq_s1_ctx* ctx);

/* Test hook: one stage-1 convolution through the decoder's own path (weight packing, tile planner, conv kernel), synchronous
 * on `stream`, device pointers.  prec: HQ_PREC_BF16 or HQ_PREC_TF32.  A: padded NHWC input [B, res+2, res+2, Cin] in the
 * operand type (bf16 | fp32; under HQ_PREC_TF32 the kernel reads it as TF32, so pass values already rounded), border zero;
 * weight fp32 [Cout, Cin, k, k] (k = 1 or 3; packed and rounded as hq_s1_load_param does); bias fp32 [Cout]; Cin a
 * multiple of 64.  mode 0: out fp32 [B, res+2, res+2, Cout], interior written, += resid (fp32, same layout, may equal
 * out) when resid != NULL; 1: out in the operand type (fp32 unrounded under HQ_PREC_TF32), interior written; 2: out fp32
 * image [B, Cout, res, res].  tile: 0 = the planner's width, else a multiple of 32 in [32, 256]. */
int hq_debug_s1_conv(int prec, const void* A, const float* weight, const float* bias, int B, int res, int Cin, int Cout,
                     int k, int mode, int tile, const float* resid, void* out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* HQGRAFT_H_ */
