"""Python handle on one libhqgraft context (one GPU).  Thin: marshals pointers, nothing numeric."""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import Dict, Optional, Sequence, Union

import torch

from . import _lib
from ._lib import HQConfig, HQRunArgs, HQSamplingParams, check

_TORCH2HQ = {torch.float32: _lib.HQ_F32, torch.bfloat16: _lib.HQ_BF16, torch.float16: _lib.HQ_F16}
# activation dtype of the debug hooks -> engine precision (bf16 / fp16: the tcgen05 engines, fp32: the CUDA-core engine)
_ACT2PREC = {torch.bfloat16: _lib.HQ_PREC_BF16, torch.float16: _lib.HQ_PREC_F16, torch.float32: _lib.HQ_PREC_FP32}


@dataclass
class SamplingParams:
    """Arguments of Sample(z; T, k, p) (hierarchical_ar.py:762-785).  None follows the reference's None."""
    top_k_top: Optional[int] = None
    top_p_top: Optional[float] = None
    top_k_bot: Optional[int] = None
    top_p_bot: Optional[float] = None
    temperature_top: float = 1.0
    temperature_bot: float = 1.0
    seed: int = 0
    row_offset: int = 0
    # middle level of the 3-level HQTransformer (top = level 0, bot = level 2 there)
    top_k_mid: Optional[int] = None
    top_p_mid: Optional[float] = None
    temperature_mid: float = 1.0

    def to_c(self) -> HQSamplingParams:
        # top_p <= 0 (not None): the reference's nucleus cut then drops every sorted entry but the first
        # (cumulative mass of the preceding entries >= 0 always, utils/sampling.py:27-31) - i.e. greedy.  The ABI
        # reserves 0 for "no cut", so that case is sent as top_k = 1.
        def k_of(k, p):
            if p is not None and float(p) <= 0.0:
                return 1
            return int(k) if k else 0
        return HQSamplingParams(
            top_k_top=k_of(self.top_k_top, self.top_p_top),
            top_k_bot=k_of(self.top_k_bot, self.top_p_bot),
            top_p_top=float(self.top_p_top) if self.top_p_top is not None else 0.0,
            top_p_bot=float(self.top_p_bot) if self.top_p_bot is not None else 0.0,
            temperature_top=float(self.temperature_top), temperature_bot=float(self.temperature_bot),
            seed=int(self.seed) & 0xFFFFFFFFFFFFFFFF, row_offset=int(self.row_offset),
            top_k_mid=k_of(self.top_k_mid, self.top_p_mid),
            top_p_mid=float(self.top_p_mid) if self.top_p_mid is not None else 0.0,
            temperature_mid=float(self.temperature_mid), reserved=0)


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


class Engine:
    """Owns an hq_ctx: parameters in engine layout, KV cache, workspaces, captured graphs."""

    def __init__(self, *, embed_dim: int, n_heads: int, n_layers: int, n_layers_depth: int, vocab_top: int,
                 vocab_bot: int, vocab_txt: int = 16384, n_classes: int = 1000, ctx_len_img: int = 256,
                 ctx_len_txt: int = 64, cond: str = "cls", precision: str = "bf16", max_seq_len: int = 64,
                 max_batch: int = 16, device: Union[int, str, torch.device] = 0, use_cuda_graph: bool = True,
                 use_pdl: bool = True, use_chain: bool = False, model_type: str = "parallel",
                 embedding_type: str = "transformer1", position_embedding: str = "1d", code_levels: int = 2,
                 vocab_mid: int = 0, fuse_head_sampler: bool = True):
        if precision not in _lib.HQ_PREC:
            raise ValueError(f"precision={precision!r}: one of {sorted(_lib.HQ_PREC)}")
        self._lib = _lib.load()
        self._ctx = C.c_void_p()
        dev = torch.device(device) if not isinstance(device, int) else torch.device("cuda", device)
        if dev.type != "cuda":
            raise ValueError("hqtransformer_b200 runs on CUDA (sm_100a) devices only; there is no CPU path")
        self.device = torch.device("cuda", dev.index or 0)
        self.cond = cond
        self.precision = precision
        self.embed_dim, self.ctx_len_txt, self.max_seq_len = embed_dim, ctx_len_txt, max_seq_len
        self.vocab_max = max(vocab_top, vocab_bot)
        cfg = HQConfig(embed_dim=embed_dim, n_heads=n_heads, n_layers=n_layers, n_layers_depth=n_layers_depth,
                       vocab_top=vocab_top, vocab_bot=vocab_bot, vocab_txt=vocab_txt, n_classes=n_classes or 0,
                       ctx_len_img=ctx_len_img, ctx_len_txt=ctx_len_txt,
                       cond_kind={"cls": _lib.HQ_COND_CLS, "txt": _lib.HQ_COND_TXT, "uncond": _lib.HQ_COND_UNCOND}[cond],
                       precision=_lib.HQ_PREC[precision],
                       max_seq_len=max_seq_len, use_cuda_graph=1 if use_cuda_graph else 0,
                       use_pdl=1 if use_pdl else 0, use_chain=1 if use_chain else 0,
                       model_type=_lib.HQ_MODEL[model_type], embedding_kind=_lib.HQ_EMB[embedding_type],
                       position_kind=_lib.HQ_POS[position_embedding], code_levels=int(code_levels), vocab_mid=int(vocab_mid),
                       fuse_head_sampler=1 if fuse_head_sampler else 0)
        self.code_levels = int(code_levels)
        if self.code_levels == 3:
            self.vocab_max = max(self.vocab_max, int(vocab_mid))
        check(self._lib.hq_create(C.byref(cfg), self.device.index, int(max_batch), C.byref(self._ctx)), None, "hq_create")

    # ---- lifetime ----
    def close(self) -> None:
        if getattr(self, "_ctx", None) is not None and self._ctx.value:
            self._lib.hq_destroy(self._ctx)
            self._ctx = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def max_batch(self) -> int:
        return self._lib.hq_max_batch(self._ctx)

    def reserve_batch(self, max_batch: int) -> None:
        check(self._lib.hq_reserve_batch(self._ctx, int(max_batch)), self._ctx, "hq_reserve_batch")

    @property
    def device_bytes(self) -> int:
        return self._lib.hq_device_bytes(self._ctx)

    @property
    def last_launch_count(self) -> int:
        return self._lib.hq_last_launch_count(self._ctx)

    @property
    def chain_launches(self) -> int:
        """Launches of the persistent chain kernel since the ctx was created (0: every op ran as its own kernel)."""
        return self._lib.hq_chain_launch_count(self._ctx)

    # ---- parameters ----
    def load_param(self, name: str, t: torch.Tensor) -> None:
        t = t.detach()
        if t.dtype not in _TORCH2HQ:
            t = t.float()
        t = t.contiguous()
        shape = (C.c_int64 * t.dim())(*t.shape)
        if t.is_cuda and t.device != self.device:
            t = t.to(self.device)
        check(self._lib.hq_load_param(self._ctx, name.encode(), t.data_ptr(), _TORCH2HQ[t.dtype], shape, t.dim(),
                                      1 if t.is_cuda else 0), self._ctx, f"hq_load_param({name})")

    def load_state_dict(self, sd: Dict[str, torch.Tensor], strict: bool = True) -> None:
        """`load_state_dict(strict=True)` semantics (sampling_hqmodel.py:79): unknown keys, wrong shapes and
        missing keys raise.  strict=False ignores unknown and missing keys only - a shape mismatch or a CUDA failure
        still raises, as torch's `load_state_dict(strict=False)` does."""
        for k, v in sd.items():
            try:
                self.load_param(k, v)
            except _lib.HQError as e:
                if strict or "unexpected key" not in str(e):
                    raise
        if strict:
            check(self._lib.hq_params_complete(self._ctx), self._ctx, "load_state_dict")

    # ---- the loop ----
    def run(self, *, batch: int, seq_len: int, pos_begin: int, pos_end: int, sampling: SamplingParams,
            cond: Optional[torch.Tensor] = None, sos: Optional[torch.Tensor] = None,
            given_top: Optional[torch.Tensor] = None, given_bot: Optional[torch.Tensor] = None,
            codes_top: torch.Tensor = None, codes_bot: torch.Tensor = None,
            logits: Optional[torch.Tensor] = None, host: bool = False, stream: Optional[int] = None,
            codes_mid: Optional[torch.Tensor] = None, given_mid: Optional[torch.Tensor] = None,
            shared_prefix: bool = False, prefix_len: int = 0) -> None:
        """hq_run (device tensors, async on the current torch stream) or hq_run_host (CPU tensors, synchronous).
        prefix_len > 0 (with pos_begin 0): image completion - codes_top / codes_bot (/ codes_mid) hold the given codes of
        positions < prefix_len, which come back unchanged; the rest is sampled after them."""
        tensors = dict(cond=cond, sos=sos, given_top=given_top, given_bot=given_bot, codes_top=codes_top,
                       codes_bot=codes_bot, logits=logits, codes_mid=codes_mid, given_mid=given_mid)
        for k, t in tensors.items():
            if t is None:
                continue
            want = torch.float32 if k in ("sos", "logits") else torch.int64
            if t.dtype != want or not t.is_contiguous():
                raise ValueError(f"{k} must be a contiguous {want} tensor")
            if host != (not t.is_cuda):
                raise ValueError(f"{k} must live on {'the host' if host else 'the GPU'} for this call")
        args = HQRunArgs(batch=batch, seq_len=seq_len, pos_begin=pos_begin, pos_end=pos_end,
                         cond=_ptr(cond), sos=_ptr(sos), given_top=_ptr(given_top), given_bot=_ptr(given_bot),
                         codes_top=_ptr(codes_top), codes_bot=_ptr(codes_bot), logits=_ptr(logits),
                         sampling=sampling.to_c(), codes_mid=_ptr(codes_mid), given_mid=_ptr(given_mid),
                         shared_prefix=1 if shared_prefix else 0, prefix_len=int(prefix_len))
        if host:
            check(self._lib.hq_run_host(self._ctx, C.byref(args)), self._ctx, "hq_run_host")
        else:
            if stream is None:
                stream = torch.cuda.current_stream(self.device).cuda_stream
            check(self._lib.hq_run(self._ctx, C.byref(args), C.c_void_p(stream)), self._ctx, "hq_run")

    def trace_run(self, *, batch: int, seq_len: int, pos_begin: int, pos_end: int, sampling: SamplingParams,
                  cond: Optional[torch.Tensor], codes_top: torch.Tensor, codes_bot: torch.Tensor,
                  max_entries: int = 16384):
        """hq_trace_run: returns [(tag, start_ns, end_ns), ...] per kernel launch of one run (device timeline)."""
        args = HQRunArgs(batch=batch, seq_len=seq_len, pos_begin=pos_begin, pos_end=pos_end, cond=_ptr(cond), sos=None,
                         given_top=None, given_bot=None, codes_top=_ptr(codes_top), codes_bot=_ptr(codes_bot),
                         logits=None, sampling=sampling.to_c())
        out = (C.c_uint64 * (2 * max_entries))()
        tags = C.create_string_buffer(48 * max_entries)
        n = C.c_int()
        st = torch.cuda.current_stream(self.device).cuda_stream
        check(self._lib.hq_trace_run(self._ctx, C.byref(args), C.c_void_p(st), out, tags, max_entries, C.byref(n)),
              self._ctx, "hq_trace_run")
        raw = tags.raw
        return [(raw[48 * i:48 * i + 48].split(b"\0")[0].decode(), int(out[2 * i]), int(out[2 * i + 1]))
                for i in range(n.value)]

    def gemm_phases(self, *, launch_id: int, batch: int, seq_len: int, pos_begin: int, pos_end: int, sampling: SamplingParams,
                    cond: Optional[torch.Tensor], codes_top: torch.Tensor, codes_bot: torch.Tensor, max_ctas: int = 160,
                    max_entries: int = 16384):
        """hq_debug_gemm_phases: (timeline as trace_run, int64 [max_ctas, 16] per-CTA phase stamps of launch `launch_id`)."""
        import numpy as np
        args = HQRunArgs(batch=batch, seq_len=seq_len, pos_begin=pos_begin, pos_end=pos_end, cond=_ptr(cond), sos=None,
                         given_top=None, given_bot=None, codes_top=_ptr(codes_top), codes_bot=_ptr(codes_bot),
                         logits=None, sampling=sampling.to_c())
        out = (C.c_uint64 * (2 * max_entries))()
        tags = C.create_string_buffer(48 * max_entries)
        ph = (C.c_uint64 * (max_ctas * 16))()
        n = C.c_int()
        st = torch.cuda.current_stream(self.device).cuda_stream
        check(self._lib.hq_debug_gemm_phases(self._ctx, C.byref(args), C.c_void_p(st), launch_id, ph, max_ctas, out, tags,
                                             max_entries, C.byref(n)), self._ctx, "hq_debug_gemm_phases")
        raw = tags.raw
        tl = [(raw[48 * i:48 * i + 48].split(b"\0")[0].decode(), int(out[2 * i]), int(out[2 * i + 1])) for i in range(n.value)]
        return tl, np.frombuffer(ph, dtype=np.uint64).reshape(max_ctas, 16).astype(np.int64)

    def bench_attention(self, batch: int, n_keys: int, iters: int = 50) -> float:
        """Mean microseconds of one single-query KV-cache attention launch (CUDA events on the current stream)."""
        us = C.c_float()
        st = torch.cuda.current_stream(self.device).cuda_stream
        check(self._lib.hq_bench_attention(self._ctx, batch, n_keys, iters, C.byref(us), C.c_void_p(st)), self._ctx,
              "hq_bench_attention")
        return us.value

    def attention_phases(self, batch: int, n_keys: int, warm: int = 3, max_ctas: int = 4096):
        """Per-CTA timestamps (ns) of one decode-attention launch: int64 array [n_ctas, 8] (hq_debug_attention_phases)."""
        import numpy as np
        buf = (C.c_uint64 * (max_ctas * 8))()
        n = C.c_int()
        st = torch.cuda.current_stream(self.device).cuda_stream
        check(self._lib.hq_debug_attention_phases(self._ctx, batch, n_keys, warm, buf, max_ctas, C.byref(n), C.c_void_p(st)),
              self._ctx, "hq_debug_attention_phases")
        return np.frombuffer(buf, dtype=np.uint64).reshape(max_ctas, 8)[:n.value].astype(np.int64)

    def chain_phases(self, *, batch: int, seq_len: int, pos_begin: int, pos_end: int, sampling: SamplingParams,
                     cond: Optional[torch.Tensor], codes_top: torch.Tensor, codes_bot: torch.Tensor, launch_idx: int,
                     op_idx: int, max_ctas: int = 256):
        """Per-CTA timestamps (ns) of one op of one persistent chain launch: int64 array [n_ctas, 8] (hq_debug_chain_phases)."""
        import numpy as np
        args = HQRunArgs(batch=batch, seq_len=seq_len, pos_begin=pos_begin, pos_end=pos_end, cond=_ptr(cond), sos=None,
                         given_top=None, given_bot=None, codes_top=_ptr(codes_top), codes_bot=_ptr(codes_bot),
                         logits=None, sampling=sampling.to_c())
        buf = (C.c_uint64 * (max_ctas * 8))()
        n = C.c_int()
        st = torch.cuda.current_stream(self.device).cuda_stream
        check(self._lib.hq_debug_chain_phases(self._ctx, C.byref(args), C.c_void_p(st), launch_idx, op_idx, buf, max_ctas,
                                              C.byref(n)), self._ctx, "hq_debug_chain_phases")
        return np.frombuffer(buf, dtype=np.uint64).reshape(max_ctas, 8)[:n.value].astype(np.int64)

    def bench_gemm(self, kind: int, M: int, iters: int = 20) -> float:
        """Mean microseconds of one GEMM launch of family `kind` (0 qkv, 1 proj, 2 fc1, 3 fc2, 4 head_top) at M rows,
        L2 evicted between launches."""
        us = C.c_float()
        st = torch.cuda.current_stream(self.device).cuda_stream
        check(self._lib.hq_bench_gemm(self._ctx, kind, M, iters, C.byref(us), C.c_void_p(st)), self._ctx,
              "hq_bench_gemm")
        return us.value


# ---- stand-alone hooks used by tests / bench ----
def debug_gemm(A: torch.Tensor, W: torch.Tensor, tile: int = 0) -> torch.Tensor:
    """C = A @ W^T through the engine's GEMM kernels (bf16 / fp16 -> tcgen05 path, fp32 -> CUDA-core path).
    tile: 0 = engine heuristic, 32..256 = CTA-pair kernel of that width, -64/-128 = single-CTA kernel."""
    lib = _lib.load()
    assert A.is_cuda and W.is_cuda and A.dtype == W.dtype and A.is_contiguous() and W.is_contiguous()
    M, K = A.shape
    N = W.shape[0]
    out = torch.empty(M, N, dtype=torch.float32, device=A.device)
    prec = _ACT2PREC[A.dtype]
    with torch.cuda.device(A.device):
        st = torch.cuda.current_stream(A.device).cuda_stream
        check(lib.hq_debug_gemm(prec, A.data_ptr(), W.data_ptr(), out.data_ptr(), M, N, K, tile, C.c_void_p(st)), None,
              "hq_debug_gemm")
    return out


EPI_QKV, EPI_RESID, EPI_GELU, EPI_F32 = 0, 1, 2, 3


def debug_gemm_epi(A: torch.Tensor, W: torch.Tensor, epi: int, *, N: Optional[int] = None, w_row_off: int = 0,
                   tile: int = 0, ks1: bool = False, bias: Optional[torch.Tensor] = None,
                   q: Optional[torch.Tensor] = None, kdst: Optional[torch.Tensor] = None, vdst: Optional[torch.Tensor] = None,
                   vdup: Optional[torch.Tensor] = None, D: int = 0, sec0: int = 0, rpb: int = 1, t_stride: int = 1, t0: int = 0,
                   x: Optional[torch.Tensor] = None, out: Optional[torch.Tensor] = None, outf: Optional[torch.Tensor] = None,
                   ldo: int = 0, splits: int = 1, split_stride: int = 0) -> None:
    """A [M, K] @ W[w_row_off : w_row_off + N]^T through the engine's GEMM kernels with fused epilogue `epi` (EPI_QKV,
    EPI_RESID, EPI_GELU or EPI_F32), writing into the caller's buffers in place; see hq_debug_epi in include/hqgraft.h.
    bf16 / fp16 A / W take the tcgen05 kernels (`tile` and `ks1` pin the plan), fp32 the CUDA-core kernel.  Synchronous."""
    lib = _lib.load()
    assert A.is_cuda and W.is_cuda and A.dtype == W.dtype and A.is_contiguous() and W.is_contiguous()
    act = A.dtype
    for t in (q, kdst, vdst, vdup, out):
        assert t is None or (t.dtype == act and t.is_contiguous() and t.device == A.device)
    for t in (bias, x, outf):
        assert t is None or (t.dtype == torch.float32 and t.is_contiguous() and t.device == A.device)
    M, K = A.shape
    w_rows = W.shape[0]
    if N is None:
        N = w_rows - w_row_off
    e = _lib.HQDebugEpi(epi=epi, tile=tile, ks1=int(bool(ks1)), D=D, sec0=sec0, rpb=rpb, t_stride=t_stride, t0=t0,
                        w_row_off=w_row_off, ldo=ldo, splits=splits, reserved=0, split_stride=split_stride,
                        bias=_ptr(bias), q=_ptr(q), kdst=_ptr(kdst), vdst=_ptr(vdst), vdup=_ptr(vdup), x=_ptr(x),
                        out=_ptr(out), outf=_ptr(outf))
    prec = _ACT2PREC[act]
    with torch.cuda.device(A.device):
        st = torch.cuda.current_stream(A.device).cuda_stream
        check(lib.hq_debug_gemm_epi(prec, A.data_ptr(), W.data_ptr(), w_rows, M, N, K, C.byref(e), C.c_void_p(st)), None,
              "hq_debug_gemm_epi")


def debug_layernorm(x: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor, out: torch.Tensor, rows: int, *,
                    add: Optional[torch.Tensor] = None, in_group: int = 1, in_mul: int = 1, in_off: int = 0,
                    out_mul: int = 1, fold: Optional[torch.Tensor] = None, n_fold: int = 0, fold_stride: int = 0,
                    fold_bias: Optional[torch.Tensor] = None) -> None:
    """The engine's LayerNorm launch (layernorm_kernel, instantiation chosen by n_fold as in the sampler) on fp32 x
    [*, D], in place: out[r * out_mul] = LN(x[(r // in_group) * in_mul + in_off + r % in_group]) * gamma + beta (+ add);
    with n_fold > 0 that x row first gets fold_bias + the partial sums fold.view(-1)[s * fold_stride + row * D ...] added
    and written back.  `out` is bf16, fp16 or fp32.  Synchronous."""
    lib = _lib.load()
    D = x.shape[-1]
    for t in (x, gamma, beta, add, fold, fold_bias):
        assert t is None or (t.is_cuda and t.dtype == torch.float32 and t.is_contiguous())
    assert out.is_contiguous() and out.dtype in _ACT2PREC
    prec = _ACT2PREC[out.dtype]
    with torch.cuda.device(x.device):
        st = torch.cuda.current_stream(x.device).cuda_stream
        check(lib.hq_debug_layernorm(prec, x.data_ptr(), gamma.data_ptr(), beta.data_ptr(), _ptr(add), out.data_ptr(), rows,
                                     D, in_group, in_mul, in_off, out_mul, _ptr(fold), n_fold, fold_stride, _ptr(fold_bias),
                                     C.c_void_p(st)), None, "hq_debug_layernorm")


def debug_attention(q: torch.Tensor, K: torch.Tensor, V: torch.Tensor, n_keys: int, variant: int = 0) -> torch.Tensor:
    """Single-query attention of every row of q [B, D] over the first n_keys rows of its cache K / V [B, T, D]
    (head size 64) through the engine's decode kernels; variant 0 = engine choice, 1 = scalar bulk-staged kernel."""
    lib = _lib.load()
    assert q.is_cuda and q.dtype == K.dtype == V.dtype and q.dtype in _ACT2PREC
    assert q.is_contiguous() and K.is_contiguous() and V.is_contiguous() and K.shape == V.shape
    B, D = q.shape
    T = K.shape[1]
    assert K.shape == (B, T, D) and D % 64 == 0 and 1 <= n_keys <= T
    out = torch.empty_like(q)
    prec = _ACT2PREC[q.dtype]
    with torch.cuda.device(q.device):
        st = torch.cuda.current_stream(q.device).cuda_stream
        check(lib.hq_debug_attention(prec, q.data_ptr(), K.data_ptr(), V.data_ptr(), out.data_ptr(), B, D // 64, T, n_keys,
                                     variant, C.c_void_p(st)), None, "hq_debug_attention")
    return out


def debug_attention_prefix(q: torch.Tensor, K: torch.Tensor, V: torch.Tensor, variant: int = 0) -> torch.Tensor:
    """Causal attention of the image-completion prefix pass: query i of q [B, n_q, D] over keys 0 .. i of K / V [B, T, D]
    (head size 64, T >= n_q) through the engine's kernel for that pass (bf16 / fp16: the tensor-core prefix kernel, fp32:
    the fp32 engine's per-query kernel); variant 1: the per-query kernel at every precision (the text prefill's)."""
    lib = _lib.load()
    assert q.is_cuda and q.dtype == K.dtype == V.dtype and q.dtype in _ACT2PREC
    assert q.is_contiguous() and K.is_contiguous() and V.is_contiguous() and K.shape == V.shape
    B, n_q, D = q.shape
    T = K.shape[1]
    assert K.shape == (B, T, D) and D % 64 == 0 and 1 <= n_q <= T
    out = torch.empty_like(q)
    with torch.cuda.device(q.device):
        st = torch.cuda.current_stream(q.device).cuda_stream
        check(lib.hq_debug_attention_prefix(_ACT2PREC[q.dtype], q.data_ptr(), K.data_ptr(), V.data_ptr(), out.data_ptr(), B,
                                            D // 64, T, n_q, int(variant), C.c_void_p(st)), None, "hq_debug_attention_prefix")
    return out


def debug_philox(seed: int, counter: Sequence[int]):
    lib = _lib.load()
    c = (C.c_uint32 * 4)(*counter)
    o = (C.c_uint32 * 4)()
    check(lib.hq_debug_philox(seed, c, o), None, "hq_debug_philox")
    return [int(v) for v in o]


def debug_sample(logits: torch.Tensor, temperature: float = 1.0, top_k: Optional[int] = None,
                 top_p: Optional[float] = None, seed: int = 0, row_offset: int = 0, position: int = 0, slot: int = 0,
                 return_probs: bool = False):
    """Sample(z; T, k, p) for each row of device logits [R, V]; returns int64 codes [R] (and probs [R, V])."""
    lib = _lib.load()
    assert logits.is_cuda and logits.dtype == torch.float32 and logits.is_contiguous() and logits.dim() == 2
    R, V = logits.shape
    codes = torch.empty(R, dtype=torch.int64, device=logits.device)
    probs = torch.empty(R, V, dtype=torch.float32, device=logits.device) if return_probs else None
    with torch.cuda.device(logits.device):
        st = torch.cuda.current_stream(logits.device).cuda_stream
        check(lib.hq_debug_sample(logits.data_ptr(), R, V, float(temperature), int(top_k) if top_k else 0,
                                  float(top_p) if top_p is not None else 0.0, seed, row_offset, position, slot,
                                  codes.data_ptr(), _ptr(probs), C.c_void_p(st)), None, "hq_debug_sample")
    return (codes, probs) if return_probs else codes


def bench_gemm_shape(M: int, N: int, K: int, tile: int = 0, iters: int = 20, flush: int = 2, copies: int = 1):
    """(mean, min) microseconds per launch of the bf16 GEMM kernel on synthetic operands (hq_bench_gemm_shape)."""
    lib = _lib.load()
    mean, mn = C.c_float(), C.c_float()
    st = torch.cuda.current_stream().cuda_stream
    check(lib.hq_bench_gemm_shape(M, N, K, tile, iters, flush, copies, C.byref(mean), C.byref(mn), C.c_void_p(st)), None,
          "hq_bench_gemm_shape")
    return mean.value, mn.value
