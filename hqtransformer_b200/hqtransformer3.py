"""3-level HQ-Transformer (SURVEY.md 8f-2): host mirror of `HQTransformer` (hqvae/models/stage2/hqtransformer.py) and
`sampling_hqtransformer` (hqvae/utils/sampling.py:240-307), sampling only, backed by libhqgraft (hq_config.code_levels = 3).

Per top position: one spatial-transformer step over the mean of the 21 stack-token embeddings, then three passes of the
depth transformer - 1 top, 4 middle, 16 bottom tokens ('parallel' mask, layers.py:154-178) - and 21 categorical draws with
one (temperature, top-k, top-p) per level.  Implemented: decoding_type 'parallel-add' (the shipped `*-level3.yaml`
configs), embedding_type 'transformer1', 1-D positions, class-conditional or unconditional `sos`.
"""
from __future__ import annotations

import copy
from collections import OrderedDict
from types import SimpleNamespace
from typing import Dict, List, Optional, Sequence, Tuple, Union

import torch

from .engine import Engine, SamplingParams
from .models import _block_shapes, fresh_seed


class HQTransformer:
    def __init__(self, vocab_sizes: Sequence[int], vocab_size_txt: int, decoding_type: Optional[str], use_cls_cond: bool,
                 use_txt_cond: bool, hparams, hparams_dec=None, *, device: Union[int, str, torch.device] = 0,
                 precision: str = "bf16", max_batch: int = 16, max_seq_len: int = 64, use_cuda_graph: bool = True,
                 use_pdl: bool = True, fuse_head_sampler: bool = True) -> None:
        if len(vocab_sizes) != 3:
            raise NotImplementedError("HQTransformer: three code levels (1 + 4 + 16 codes per position) are implemented")
        if decoding_type != "parallel-add":
            raise NotImplementedError(f"decoding_type={decoding_type!r}: only 'parallel-add' is implemented "
                                      "('tree', 'top2mid2bot' and the 'reduce' variants are not)")
        if use_txt_cond:
            raise NotImplementedError("text-conditional 3-level models are not implemented")
        if getattr(hparams, "embedding_type", "transformer1") != "transformer1" or getattr(hparams, "position_embedding", "1d") != "1d":
            raise NotImplementedError("HQTransformer: embedding_type 'transformer1' with position_embedding '1d' only")
        if hparams_dec is None:                                   # hqtransformer.py:204-208
            hparams_dec = copy.deepcopy(hparams)
            hparams_dec.n_layers = 4
        if hparams_dec.embed_dim != hparams.embed_dim or hparams_dec.n_heads != hparams.n_heads:
            raise NotImplementedError("depth transformer must share embed_dim / n_heads with the spatial transformer")
        self.vocab_sizes = [int(v) for v in vocab_sizes]
        self.vocab_size_txt = vocab_size_txt
        self.use_cls_cond, self.use_txt_cond = bool(use_cls_cond), False
        self.decoding_type = decoding_type
        self.code_level, self.code_len, self.num_pairs = 3, 21, 4
        self.idx_pred = 0
        self.ctx_len_img = hparams.ctx_len_img
        self.n_layers, self.n_layers_depth = hparams.n_layers, hparams_dec.n_layers
        self.embed_dim, self.n_heads = hparams.embed_dim, hparams.n_heads
        self.n_classes = getattr(hparams, "n_classes", None)
        self.cond = "cls" if self.use_cls_cond else "uncond"
        self.device = torch.device(device) if not isinstance(device, int) else torch.device("cuda", device)
        self.precision = precision
        self.max_seq_len = min(max_seq_len, self.ctx_len_img)
        self._engine_kw = dict(embed_dim=self.embed_dim, n_heads=self.n_heads, n_layers=self.n_layers,
                               n_layers_depth=self.n_layers_depth, vocab_top=self.vocab_sizes[0], vocab_bot=self.vocab_sizes[2],
                               vocab_mid=self.vocab_sizes[1], code_levels=3, n_classes=self.n_classes or 0,
                               ctx_len_img=self.ctx_len_img, cond=self.cond, max_seq_len=self.max_seq_len,
                               device=self.device, use_cuda_graph=use_cuda_graph, use_pdl=use_pdl,
                               fuse_head_sampler=fuse_head_sampler)
        self._max_batch = max_batch
        self._engines: Dict[str, Engine] = {}
        self._source = None
        self.training = False
        self.engine(precision)

    def engine(self, precision: Optional[str] = None) -> Engine:
        precision = precision or self.precision
        if precision not in self._engines:
            eng = Engine(precision=precision, max_batch=self._max_batch, **self._engine_kw)
            if self._source is not None:
                eng.load_state_dict(self._source, strict=True)
            elif self._engines:
                raise RuntimeError(f"no {precision} engine: load_state_dict(..., keep_source=True) is needed to re-pack weights")
            self._engines[precision] = eng
        return self._engines[precision]

    def _engine_for(self, use_fp16: bool, batch: int) -> Engine:
        # use_fp16=True: the model's 2-byte engine - fp16 when it was built with precision="fp16", bf16 otherwise
        eng = self.engine(("fp16" if self.precision == "fp16" else "bf16") if use_fp16 else "fp32")
        if batch > eng.max_batch:
            eng.reserve_batch(batch)
        return eng

    def eval(self):
        self.training = False
        return self

    def to(self, device):
        return self

    def param_shapes(self) -> "OrderedDict[str, Tuple[int, ...]]":
        """Every key `load_state_dict(strict=True)` requires (hqtransformer.py:24-166)."""
        D = self.embed_dim
        s: "OrderedDict[str, Tuple[int, ...]]" = OrderedDict()
        for i, v in enumerate(self.vocab_sizes):
            s[f"tok_emb_levels.{i}.weight"] = (v, D)
        s["pos_emb_emb.weight"] = (21, D)
        if self.use_cls_cond:
            s["sos.weight"] = (self.n_classes, D)
        else:
            s["sos"] = (1, 1, D)
        s["pos_emb_top.weight"] = (self.ctx_len_img, D)
        for i in range(self.n_layers):
            s.update(_block_shapes(f"blocks.{i}", D))
        s["ln_f.weight"] = (D,)
        s["ln_f.bias"] = (D,)
        s["sos_depth"] = (1, 1, D)
        for i, v in enumerate(self.vocab_sizes):
            s[f"tok_emb_depth_levels.{i}.weight"] = (v, D)
        s["pos_emb_depths.0.weight"] = (4, D)
        s["pos_emb_depths.1.weight"] = (16, D)
        for i in range(self.n_layers_depth):
            s.update(_block_shapes(f"depths.{i}", D))
        for i in range(3):
            s[f"ln_levels.{i}.weight"] = (D,)
            s[f"ln_levels.{i}.bias"] = (D,)
        for i, v in enumerate(self.vocab_sizes):
            s[f"head_levels.{i}.weight"] = (v, D)
        return s

    def load_state_dict(self, state_dict, strict: bool = True, keep_source: bool = False):
        self._source = dict(state_dict) if keep_source else None
        for eng in self._engines.values():
            eng.load_state_dict(state_dict, strict=strict)
        return SimpleNamespace(missing_keys=[], unexpected_keys=[])

    @torch.no_grad()
    def init_weights(self, seed: int = 0) -> None:
        """`HQTransformer._init_weights` statistics (hqtransformer.py:217-224), generated on the GPU."""
        g = torch.Generator(device=self.device).manual_seed(seed)
        for name, shape in self.param_shapes().items():
            leaf = name.split(".")[-1]
            is_ln = (".ln" in name or name.startswith("ln_"))
            if name in ("sos", "sos_depth"):
                t = torch.randn(shape, generator=g, device=self.device)
            elif is_ln:
                t = torch.ones(shape, device=self.device) if leaf == "weight" else torch.zeros(shape, device=self.device)
            elif leaf == "bias":
                t = torch.zeros(shape, device=self.device)
            else:
                t = torch.randn(shape, generator=g, device=self.device) * 0.02
            for eng in self._engines.values():
                eng.load_param(name, t)
            del t

    def build_cond(self, cond, num_candidates: int) -> Optional[torch.Tensor]:
        if not self.use_cls_cond:
            return None
        if isinstance(cond, int):
            if not 0 <= cond < self.n_classes:
                raise IndexError(f"class id {cond} out of range [0, {self.n_classes})")
            return torch.full((num_candidates,), cond, dtype=torch.int64, device=self.device)
        c = torch.as_tensor(cond, dtype=torch.int64).reshape(-1).to(self.device)
        if c.numel() and (int(c.min()) < 0 or int(c.max()) >= self.n_classes):
            raise IndexError(f"class ids out of range [0, {self.n_classes})")
        return c.repeat(num_candidates) if c.numel() == 1 else c


def _triple(v, name):
    if v is None:
        return [None, None, None]
    if isinstance(v, (int, float)):
        return [v, v, v]
    v = list(v)
    if len(v) != 3:
        raise ValueError(f"{name} must have one entry per code level (3), got {len(v)}")
    return v


@torch.no_grad()
def sampling_hqtransformer(model: HQTransformer, num_candidates: int, cond, top_k: Optional[List[float]] = None,
                           top_p: Optional[List[float]] = None, softmax_temperature: List[float] = [1.0, 1.0, 1.0],
                           is_tqdm: bool = True, use_fp16: bool = True, max_seq_len: int = 256, model_stage1=None, *,
                           seed: Optional[int] = None, row_offset: int = 0, prefix_codes: Optional[Sequence] = None,
                           shared_prefix: Optional[bool] = None) -> List[torch.Tensor]:
    """utils/sampling.py:240-307: returns [codes_top [B,S], codes_mid [B,S,4], codes_bot [B,S,16]] (int64).  `top_k`,
    `top_p`, `softmax_temperature`: one entry per level (hqtransformer.py:626-631).  `cond` may be a per-row class tensor.
    prefix_codes = (top [B or 1, P], mid [B or 1, P, 4], bot [B or 1, P, 16]): image completion, as `sampling_ihqgpt`'s
    prefix_code_top / prefix_code_bot - positions < P given and returned unchanged, the rest sampled after them.
    shared_prefix: every row has the same condition and prefix (None = detect; results are identical either way)."""
    if max_seq_len > model.max_seq_len:
        raise ValueError(f"max_seq_len={max_seq_len} exceeds the engine's {model.max_seq_len} top positions")
    k, p, t = _triple(top_k, "top_k"), _triple(top_p, "top_p"), _triple(softmax_temperature, "softmax_temperature")
    cond_t = model.build_cond(cond, num_candidates)
    B = cond_t.shape[0] if cond_t is not None else num_candidates
    eng = model._engine_for(use_fp16, B)
    sp = SamplingParams(top_k_top=k[0], top_p_top=p[0], top_k_bot=k[2], top_p_bot=p[2], temperature_top=float(t[0]),
                        temperature_bot=float(t[2]), top_k_mid=k[1], top_p_mid=p[1], temperature_mid=float(t[1]),
                        seed=fresh_seed() if seed is None else seed, row_offset=row_offset)
    dev = model.device
    ct = torch.empty(B, max_seq_len, dtype=torch.int64, device=dev)
    cm = torch.empty(B, max_seq_len, 4, dtype=torch.int64, device=dev)
    cb = torch.empty(B, max_seq_len, 16, dtype=torch.int64, device=dev)
    P = 0
    if prefix_codes is not None:
        from .sampling import _rows_equal, prefix_rows
        if len(prefix_codes) != 3:
            raise ValueError(f"prefix_codes must be (top, mid, bot), got {len(prefix_codes)} tensors")
        V = model.vocab_sizes
        parts = prefix_rows([(prefix_codes[0], "prefix_codes[0]", V[0], ()), (prefix_codes[1], "prefix_codes[1]", V[1], (4,)),
                             (prefix_codes[2], "prefix_codes[2]", V[2], (16,))], B, max_seq_len, dev)
        P = parts[0].shape[1]
        for dst, src in zip((ct, cm, cb), parts):
            dst[:, :P] = src
        if shared_prefix is None:
            shared_prefix = B > 1 and _rows_equal(cond_t) and all(_rows_equal(t) for t in parts)
    eng.run(batch=B, seq_len=max_seq_len, pos_begin=0, pos_end=max_seq_len, sampling=sp, cond=cond_t, codes_top=ct,
            codes_mid=cm, codes_bot=cb, prefix_len=P, shared_prefix=bool(shared_prefix) and P > 0)
    return [ct, cm, cb]


@torch.no_grad()
def step_logits3(model: HQTransformer, cond, codes: Sequence[torch.Tensor], use_fp16: bool = True) -> torch.Tensor:
    """Teacher-forced raw head outputs [B, S, 21, Vmax] for given code grids (parity hook)."""
    ct, cm, cb = [c.to(device=model.device, dtype=torch.int64).contiguous() for c in codes]
    B, S = ct.shape
    cond_t = model.build_cond(cond, B)
    eng = model._engine_for(use_fp16, B)
    logits = torch.zeros(B, S, 21, eng.vocab_max, dtype=torch.float32, device=model.device)
    eng.run(batch=B, seq_len=S, pos_begin=0, pos_end=S, sampling=SamplingParams(), cond=cond_t, given_top=ct, given_mid=cm,
            given_bot=cb, codes_top=ct.clone(), codes_mid=cm.clone(), codes_bot=cb.clone(), logits=logits)
    return logits
