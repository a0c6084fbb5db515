"""Drop-in replacements for the functions of hqvae/utils/sampling.py that sit on the HQ sampling path.

`sampling_ihqgpt` keeps the reference signature (utils/sampling.py:164-177) and return value
(codes_top int64 [B, S], codes_bot int64 [B, S, 4]); the 64-position loop, KV cache, depth passes and
draws all run inside libhqgraft (one hq_run call, replayed as a CUDA graph).
"""
from __future__ import annotations

from typing import List, Optional, Tuple

import torch

from .engine import SamplingParams, debug_sample
from .models import _temps, fresh_seed


@torch.no_grad()
def sampling_ihqgpt(model, num_candidates: int, cond, top_k_top: Optional[float] = None,
                    top_p_top: Optional[float] = None, top_k_bot: Optional[float] = None,
                    top_p_bot: Optional[float] = None, softmax_temperature: List[float] = [1.0, 1.0],
                    is_tqdm: bool = True, use_fp16: bool = True, max_seq_len: int = 256, model_stage1=None,
                    given_top_code: Optional[torch.Tensor] = None, *, seed: Optional[int] = None,
                    row_offset: int = 0, shared_prefix: Optional[bool] = None,
                    prefix_code_top: Optional[torch.Tensor] = None,
                    prefix_code_bot: Optional[torch.Tensor] = None) -> Tuple[torch.Tensor, torch.Tensor]:
    """utils/sampling.py:164-237.

    cond: class id (int, broadcast to the batch as in the reference :183-186, or an int64 [B] tensor for per-row
    classes), text ids int64 [B, ctx_len_txt], or None for unconditional models.  For text models the batch is
    `cond.shape[0]` (the reference ignores num_candidates there too).
    `is_tqdm` / `model_stage1` are accepted and unused (no per-position host loop exists to decorate).
    seed: Philox key of the draws.  Default: a fresh 63-bit value drawn from torch's default CPU generator on every
    call - like the reference's `torch.multinomial`, consecutive calls advance the global generator (the scripts call
    the sampler many times per class with identical arguments, sampling_hqmodel.py:180-193) and `set_seed`
    (utils/utils.py:6-10) reproduces the whole run.
    shared_prefix (text models): one prompt sampled B times (the reference notebook repeats a prompt 8x) - the 64-token
    prefill runs once and its KV-cache rows are broadcast.  None = detect (all rows of `cond` equal); results are
    identical either way.
    prefix_code_top [B or 1, P] / prefix_code_bot [B or 1, P, 4] (together, raster layout of the returned grids; a [1, ...]
    row is broadcast over the batch): image completion - positions < P are given and returned unchanged, positions >= P
    are sampled as the loop samples them after those codes (the same Philox counters: completing a grid's own prefix with
    its seed re-draws the same stream).  The prefix goes through the spatial transformer in one causal pass.
    `given_top_code` applies at positions >= P.  shared_prefix then means: every row has the same condition and the same
    prefix (None = detect)."""
    if max_seq_len > model.max_seq_len:
        raise ValueError(f"max_seq_len={max_seq_len} exceeds the engine's {model.max_seq_len} top positions "
                         "(the scripts pass 64 for 8x8 top codes)")
    cond_t = model.build_sos(cond, num_candidates)
    B = cond_t.shape[0] if cond_t is not None else num_candidates
    eng = model._engine_for(use_fp16, B)
    t_top, t_bot = _temps(softmax_temperature)
    sp = SamplingParams(top_k_top, top_p_top, top_k_bot, top_p_bot, t_top, t_bot,
                        seed=fresh_seed() if seed is None else seed, row_offset=row_offset)
    dev = model.device
    codes_top = torch.empty(B, max_seq_len, dtype=torch.int64, device=dev)
    codes_bot = torch.empty(B, max_seq_len, 4, dtype=torch.int64, device=dev)
    given = None
    if given_top_code is not None:
        given = given_top_code[:, :max_seq_len].to(device=dev, dtype=torch.int64)
        if given.shape[0] == 1 and B > 1:          # the reference broadcasts a [1, S] grid over the batch (:771-772)
            given = given.expand(B, -1)
        given = given.contiguous()
        if tuple(given.shape) != (B, max_seq_len):
            raise ValueError(f"given_top_code must be [B, >= {max_seq_len}], got {tuple(given_top_code.shape)}")
        if int(given.min()) < 0 or int(given.max()) >= model.vocab_size_top:
            raise IndexError(f"given_top_code out of range [0, {model.vocab_size_top})")
    P = 0
    if prefix_code_top is not None or prefix_code_bot is not None:
        if prefix_code_top is None or prefix_code_bot is None:
            raise ValueError("prefix_code_top and prefix_code_bot go together")
        pt, pb = prefix_rows([(prefix_code_top, "prefix_code_top", model.vocab_size_top, ()),
                              (prefix_code_bot, "prefix_code_bot", model.vocab_size_bot, (4,))], B, max_seq_len, dev)
        P = pt.shape[1]
        codes_top[:, :P] = pt
        codes_bot[:, :P] = pb
        if shared_prefix is None:
            shared_prefix = B > 1 and _rows_equal(cond_t) and _rows_equal(pt) and _rows_equal(pb)
    if shared_prefix is None:
        shared_prefix = bool(model.use_txt_cond and cond_t is not None and B > 1 and bool((cond_t == cond_t[:1]).all()))
    eng.run(batch=B, seq_len=max_seq_len, pos_begin=0, pos_end=max_seq_len, sampling=sp, cond=cond_t,
            given_top=given, codes_top=codes_top, codes_bot=codes_bot, shared_prefix=bool(shared_prefix), prefix_len=P)
    return codes_top, codes_bot


def _rows_equal(t: Optional[torch.Tensor]) -> bool:
    return t is None or bool((t == t[:1]).all())


def prefix_rows(parts, B: int, max_seq_len: int, dev) -> List[torch.Tensor]:
    """Checks the prefix code tensors of an image completion and returns them as int64 [B, P, ...] on `dev`.
    parts: (tensor [B or 1, P, *tail], name, vocabulary size, tail) per code level; every level must have the same P, with
    1 <= P < max_seq_len.  A [1, ...] tensor is broadcast over the batch."""
    out, P = [], None
    for t, name, vocab, tail in parts:
        t = torch.as_tensor(t)
        want = "[B or 1, P" + "".join(f", {w}" for w in tail) + "]"
        if t.dim() != 2 + len(tail) or tuple(t.shape[2:]) != tuple(tail) or t.shape[0] not in (1, B):
            raise ValueError(f"{name} must be {want} with B = {B}, got {tuple(t.shape)}")
        if t.dtype.is_floating_point or t.dtype.is_complex or t.dtype == torch.bool:
            raise ValueError(f"{name} must hold integer codes, got {t.dtype}")
        if P is None:
            P = t.shape[1]
            if not 1 <= P < max_seq_len:
                raise ValueError(f"prefix length {P} outside [1, max_seq_len={max_seq_len})")
        elif t.shape[1] != P:
            raise ValueError(f"{name} covers {t.shape[1]} positions, the other prefix tensors {P}")
        t = t.to(device=dev, dtype=torch.int64)
        if int(t.min()) < 0 or int(t.max()) >= vocab:
            raise IndexError(f"{name} out of range [0, {vocab})")
        out.append(t.expand(B, *t.shape[1:]).contiguous())
    return out


def encode_prompts(tokenizer, texts, context_length: int = 64) -> torch.Tensor:
    """Text front-end of the txt2img scripts (hqvae/datasets/__init__.py:145-152, sampling_hqmodel_txt2img.py): pad with
    "[PAD]" / truncate every prompt to `context_length` tokens with a HuggingFace `tokenizers` tokenizer built as
    hqvae/tokenizers/__init__.py:15-38 does (`create_tokenizer('bpe16k_huggingface', lowercase=True, dropout=None)`; the
    vocabulary files ship with the reference, not with this repo).  Returns int64 [len(texts), context_length]: the `cond`
    of `sampling_ihqgpt` for a text-conditional model."""
    tokenizer.add_special_tokens(["[PAD]"])
    tokenizer.enable_padding(length=context_length, pad_id=tokenizer.token_to_id("[PAD]"))
    tokenizer.enable_truncation(max_length=context_length)
    if isinstance(texts, str):
        texts = [texts]
    return torch.tensor([tokenizer.encode(t).ids for t in texts], dtype=torch.int64)


@torch.no_grad()
def step_logits(model, cond, codes_top: torch.Tensor, codes_bot: torch.Tensor, use_fp16: bool = True) -> torch.Tensor:
    """Teacher-forced raw head outputs [B, S, 5, V] (slot 0 = top, 1..4 = bottom) for given code grids - the logits
    `sampling_step` computes at every position when it emits exactly these codes.  Parity hook."""
    B, S = codes_top.shape
    cond_t = model.build_sos(cond, B)
    eng = model._engine_for(use_fp16, B)
    dev = model.device
    ct = codes_top.to(device=dev, dtype=torch.int64).contiguous()
    cb = codes_bot.to(device=dev, dtype=torch.int64).contiguous()
    if int(ct.min()) < 0 or int(ct.max()) >= model.vocab_size_top or int(cb.min()) < 0 or int(cb.max()) >= model.vocab_size_bot:
        raise IndexError("code indices out of the vocabulary range")
    out_t, out_b = ct.clone(), cb.clone()
    logits = torch.zeros(B, S, 5, eng.vocab_max, dtype=torch.float32, device=dev)
    eng.run(batch=B, seq_len=S, pos_begin=0, pos_end=S, sampling=SamplingParams(), cond=cond_t, given_top=ct,
            given_bot=cb, codes_top=out_t, codes_bot=out_b, logits=logits)
    return logits


def cutoff_topk_logits(logits: torch.Tensor, k: Optional[int]) -> torch.Tensor:
    """utils/sampling.py:12-19 on device logits [R, V]: logits below the k-th largest -> -inf (ties kept)."""
    if k is None:
        return logits
    _, probs = debug_sample(logits.float().contiguous(), 1.0, k, None, return_probs=True)
    if k == 1:  # greedy fast path reports a one-hot; the reference keeps every tie of the maximum
        return logits.masked_fill(logits < logits.max(dim=-1, keepdim=True).values, float("-inf"))
    return logits.masked_fill(probs == 0, float("-inf"))


def cutoff_topp_probs(probs: torch.Tensor, p: Optional[float]) -> torch.Tensor:
    """utils/sampling.py:22-37 on device probabilities [R, V]: nucleus cut + renormalisation."""
    if p is None:
        return probs
    _, out = debug_sample(torch.log(probs.float()).contiguous(), 1.0, None, p, return_probs=True)
    return out


def get_positional_encoding(inputs: torch.Tensor, mode: str = "1d") -> torch.Tensor:
    """utils/sampling.py:40-52 ('1d'): arange(N) repeated over the batch.  The engine derives positions itself."""
    if mode != "1d":
        raise ValueError("%s positional encoding invalid" % mode)
    B, N = inputs.shape
    return torch.arange(N, device=inputs.device).repeat((B, 1))


def grids_to_codes(codes_t: torch.Tensor, codes_b: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
    """The exact inverse of `codes_to_grids`: code grids as the reference's `stage1.get_codes` returns them, top [B, H, W]
    and bottom [B, 2H, 2W], -> the sampler's raster layout codes_top [B, H*W], codes_bot [B, H*W, 4] (within-stack order
    kh*2 + kw) - e.g. the prefix of an image completion."""
    if codes_t.dim() != 3 or codes_b.dim() != 3 or codes_b.shape[0] != codes_t.shape[0] or \
            tuple(codes_b.shape[1:]) != (2 * codes_t.shape[1], 2 * codes_t.shape[2]):
        raise ValueError(f"grids must be top [B, H, W] and bottom [B, 2H, 2W], got {tuple(codes_t.shape)} and "
                         f"{tuple(codes_b.shape)}")
    B, H, W = codes_t.shape
    top = codes_t.reshape(B, H * W)
    bot = codes_b.reshape(B, H, 2, W, 2).permute(0, 1, 3, 2, 4).reshape(B, H * W, 4)
    return top, bot


def codes_to_grids(codes_top: torch.Tensor, codes_bot: torch.Tensor, H: int = 8) -> Tuple[torch.Tensor, torch.Tensor]:
    """HQ-VAE code layout consumed by `stage1.decode_code` (sampling_hqmodel.py:119-120):
    'B (H W) -> B H W' and 'B (H W) (kerH kerW) -> B (H kerH) (W kerW)', kerH = kerW = 2."""
    B = codes_top.shape[0]
    W = codes_top.shape[1] // H
    top = codes_top.reshape(B, H, W)
    bot = codes_bot.reshape(B, H, W, 2, 2).permute(0, 1, 3, 2, 4).reshape(B, 2 * H, 2 * W)
    return top, bot
