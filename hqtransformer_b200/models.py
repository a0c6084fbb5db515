"""Host-side mirror of the reference's stage-2 model objects for the sampling path.

`iHQGPT` takes the reference constructor's arguments (hqvae/models/stage2/hierarchical_ar.py:24-33),
accepts the reference `state_dict` (same key names, strict), and exposes `sampling_step` with the
reference signature (:428-443).  It owns no torch parameters: weights live in the libhqgraft engine.
`ImageGPT2` mirrors the wrapper the scripts build (hqvae/models/__init__.py:92-174, 207-215).
"""
from __future__ import annotations

import copy
import math
from collections import OrderedDict
from types import SimpleNamespace
from typing import Dict, List, Optional, Tuple, Union

import torch

from .config import engine_kwargs, load_config
from .engine import Engine, SamplingParams


def _temps(softmax_temperature) -> Tuple[float, float]:
    """The reference indexes softmax_temperature[0/1] (hierarchical_ar.py:763, 779); measure_throughput_txt passes a
    bare float (:135), which raises there - accept both."""
    if isinstance(softmax_temperature, (int, float)):
        return float(softmax_temperature), float(softmax_temperature)
    return float(softmax_temperature[0]), float(softmax_temperature[1])


def fresh_seed() -> int:
    """Philox key for one sampling call: 63 random bits from torch's default CPU generator.  Every call advances that
    generator (as `torch.multinomial` does in the reference), so two consecutive default calls draw different
    samples, and `set_seed` / `torch.manual_seed` reproduces the whole sequence of calls."""
    return int(torch.empty((), dtype=torch.int64).random_())


def _block_shapes(prefix: str, D: int) -> "OrderedDict[str, Tuple[int, ...]]":
    s = OrderedDict()
    for ln in ("ln1", "ln2"):
        s[f"{prefix}.{ln}.weight"] = (D,)
        s[f"{prefix}.{ln}.bias"] = (D,)
    for nm in ("key", "query", "value", "proj"):                 # layers.py:43-52
        s[f"{prefix}.attn.{nm}.weight"] = (D, D)
        s[f"{prefix}.attn.{nm}.bias"] = (D,)
    s[f"{prefix}.mlp.0.weight"] = (4 * D, D)                     # layers.py:312-317
    s[f"{prefix}.mlp.0.bias"] = (4 * D,)
    s[f"{prefix}.mlp.2.weight"] = (D, 4 * D)
    s[f"{prefix}.mlp.2.bias"] = (D,)
    return s


class iHQGPT:
    """2-level HQ-Transformer, sampling only, model_type='parallel' (the shipped checkpoints' type)."""

    def __init__(self, vocab_size_top: int, vocab_size_bot: int, vocab_size_txt: int, ratio_bot2top: int,
                 use_cls_cond: bool, use_txt_cond: bool, model_type: str, hparams, hparams_dec=None, *,
                 device: Union[int, str, torch.device] = 0, precision: str = "bf16", max_batch: int = 16,
                 max_seq_len: int = 64, use_cuda_graph: bool = True, use_pdl: bool = True,
                 use_chain: bool = False, fuse_head_sampler: bool = True) -> None:
        if model_type not in ("parallel", "top2bot", "bidirectional"):
            raise NotImplementedError(
                f"model_type={model_type!r}: 'parallel', 'top2bot' and 'bidirectional' with a 2x2 bottom window are "
                "implemented (hierarchical_ar.py:40-57 also parses 'parallel<N>' / 'bidirectional<N>' window sizes)")
        if ratio_bot2top != 4:
            raise NotImplementedError("ratio_bot2top must be 4 (8x8 top + 16x16 bottom codes)")
        emb = getattr(hparams, "embedding_type", "transformer1")
        pos_emb = getattr(hparams, "position_embedding", "1d")
        if emb not in ("transformer1", "reduce") or pos_emb not in ("1d", "2d"):
            raise NotImplementedError(
                f"embedding_type={emb!r} / position_embedding={pos_emb!r}: 'transformer1' | 'reduce' with '1d' | '2d' are "
                "implemented ('baseline', 'multiple' and 'transformer<N>' with N > 1 embedding blocks are not)")
        if getattr(hparams, "use_random_order", False):
            raise NotImplementedError("use_random_order=True is not implemented")
        self.embedding_type, self.position_embedding = emb, pos_emb
        if getattr(hparams, "gelu_use_approx", False):
            raise NotImplementedError("gelu_use_approx=True is not implemented (shipped configs use exact erf GELU)")
        if hparams_dec is None:                                   # hierarchical_ar.py:150-153
            hparams_dec = copy.deepcopy(hparams)
            hparams_dec.n_layers = 4
        if hparams_dec.embed_dim != hparams.embed_dim or hparams_dec.n_heads != hparams.n_heads:
            raise NotImplementedError("depth transformer must share embed_dim / n_heads with the spatial transformer")
        self.use_cls_cond, self.use_txt_cond = bool(use_cls_cond), bool(use_txt_cond)
        self.model_type = model_type
        self.bot_win = 1 if model_type == "top2bot" else 2          # hierarchical_ar.py:40-59
        self.num_bottom_pred, self.ratio_bot2top = self.bot_win * self.bot_win, ratio_bot2top
        self.len_seq_depth = 1 + ratio_bot2top // self.num_bottom_pred
        self.top_win = int(math.sqrt(ratio_bot2top)) // self.bot_win
        self.idx_pred = hparams.ctx_len_txt if (self.use_txt_cond and not self.use_cls_cond) else 0
        self.ctx_len_img = hparams.ctx_len_img
        self.n_layers, self.n_layers_depth = hparams.n_layers, hparams_dec.n_layers
        self.embed_dim, self.n_heads = hparams.embed_dim, hparams.n_heads
        self.vocab_size_top, self.vocab_size_bot, self.vocab_size_txt = vocab_size_top, vocab_size_bot, vocab_size_txt
        self.n_classes = getattr(hparams, "n_classes", None)
        self.ctx_len_txt = hparams.ctx_len_txt
        self.cond = "cls" if self.use_cls_cond else ("txt" if self.use_txt_cond else "uncond")
        self.device = torch.device(device) if not isinstance(device, int) else torch.device("cuda", device)
        self.precision = precision
        self.max_seq_len = min(max_seq_len, self.ctx_len_img)
        self._engine_kw = dict(embed_dim=self.embed_dim, n_heads=self.n_heads, n_layers=self.n_layers,
                               n_layers_depth=self.n_layers_depth, vocab_top=vocab_size_top, vocab_bot=vocab_size_bot,
                               vocab_txt=vocab_size_txt, n_classes=self.n_classes or 0, ctx_len_img=self.ctx_len_img,
                               ctx_len_txt=self.ctx_len_txt, cond=self.cond, max_seq_len=self.max_seq_len,
                               device=self.device, use_cuda_graph=use_cuda_graph, use_pdl=use_pdl,
                               use_chain=use_chain, model_type=model_type, embedding_type=emb, position_embedding=pos_emb,
                               fuse_head_sampler=fuse_head_sampler)
        self._max_batch = max_batch
        self._engines: Dict[str, Engine] = {}
        self._source: Optional[Dict[str, torch.Tensor]] = None    # retained only when asked (other-precision engine)
        self._step_state: Optional[dict] = None
        self.training = False
        self.engine(precision)

    # ---- engine management ----
    def engine(self, precision: Optional[str] = None) -> Engine:
        precision = precision or self.precision
        if precision not in self._engines:
            eng = Engine(precision=precision, max_batch=self._max_batch, **self._engine_kw)
            if self._source is not None:
                eng.load_state_dict(self._source, strict=True)
            elif self._engines:
                raise RuntimeError(
                    f"no {precision} engine: weights were loaded without keep_source=True, so they cannot be re-packed; "
                    f"build the model with precision={precision!r} or call load_state_dict(..., keep_source=True)")
            self._engines[precision] = eng
        return self._engines[precision]

    def _engine_for(self, use_fp16: bool, batch: int) -> Engine:
        # use_fp16=True: the model's 2-byte engine - fp16 when it was built with precision="fp16", bf16 otherwise
        eng = self.engine(("fp16" if self.precision == "fp16" else "bf16") if use_fp16 else "fp32")
        if batch > eng.max_batch:
            eng.reserve_batch(batch)
        return eng

    # ---- nn.Module-compatible surface used by the scripts ----
    def eval(self):
        self.training = False
        return self

    def to(self, device):
        if torch.device(device).type != "cuda":
            raise ValueError("hqtransformer_b200 models live on CUDA devices only")
        return self

    def cuda(self, device=None):
        return self

    def param_shapes(self) -> "OrderedDict[str, Tuple[int, ...]]":
        """Every key `load_state_dict(strict=True)` requires, with its shape (hierarchical_ar.py:63-209)."""
        D = self.embed_dim
        s: "OrderedDict[str, Tuple[int, ...]]" = OrderedDict()
        if self.cond == "cls":
            s["sos.weight"] = (self.n_classes, D)
        elif self.cond == "txt":
            s["tok_emb_txt.weight"] = (self.vocab_size_txt, D)
            s["pos_emb_txt.weight"] = (self.ctx_len_txt, D)
            s["head_txt.weight"] = (self.vocab_size_txt, D)
            s["ln_txt.weight"] = (D,)
            s["ln_txt.bias"] = (D,)
        else:
            s["sos"] = (1, 1, D)
        s["sos_depth"] = (1, 1, D)
        s["tok_emb_top.weight"] = (self.vocab_size_top, D)
        if self.embedding_type == "reduce":                       # hierarchical_ar.py:85-88
            s["tok_emb_bot.weight"] = (self.vocab_size_bot, D // 4)
        else:
            s["tok_emb_bot.weight"] = (self.vocab_size_bot, D)
            s["pos_emb_emb.weight"] = (5, D)
        if self.position_embedding == "2d":                       # :121-125
            H = int(math.sqrt(self.ctx_len_img))
            s["pos_emb_top_h.weight"] = (H, D)
            s["pos_emb_top_w.weight"] = (H, D)
        else:
            s["pos_emb_top.weight"] = (self.ctx_len_img, D)
        for i in range(self.n_layers):
            s.update(_block_shapes(f"blocks.{i}", D))
        s["ln_f.weight"] = (D,)
        s["ln_f.bias"] = (D,)
        s["tok_emb_top_depth.weight"] = (self.vocab_size_top, D)
        s["tok_emb_bot_depth.weight"] = (self.vocab_size_bot, D)
        s["pos_emb_depth.weight"] = (5, D)
        for i in range(self.n_layers_depth):
            s.update(_block_shapes(f"depths.{i}", D))
        for nm, V in (("top", self.vocab_size_top), ("bot", self.vocab_size_bot)):
            s[f"ln_{nm}.weight"] = (D,)
            s[f"ln_{nm}.bias"] = (D,)
            s[f"head_{nm}.weight"] = (V, D)
        return s

    def load_state_dict(self, state_dict: Dict[str, torch.Tensor], strict: bool = True, keep_source: bool = False):
        self._source = dict(state_dict) if keep_source else None
        for eng in self._engines.values():
            eng.load_state_dict(state_dict, strict=strict)
        return SimpleNamespace(missing_keys=[], unexpected_keys=[])

    @torch.no_grad()
    def init_weights(self, seed: int = 0) -> None:
        """Random weights with the statistics of `iHQGPT._init_weights` (hierarchical_ar.py:218-225): Linear / Embedding
        N(0, 0.02), biases 0, LayerNorm (1, 0), sos_depth / uncond sos ~ N(0, 1).  Generated on the GPU, one tensor at
        a time - what `measure_throughput` gets by building the model without a checkpoint (:25-31)."""
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

    # ---- reference API: one top position ----
    @torch.no_grad()
    def sampling_step(self, sos: torch.Tensor, codes_t: Optional[torch.Tensor], codes_b: Optional[torch.Tensor],
                      pos_codes: Optional[torch.Tensor], use_fp16: bool = True,
                      top_k_top=None, top_p_top=None, top_k_bot=None, top_p_bot=None,
                      softmax_temperature=[1.0, 1.0], past=None, model_stage1=None, given_top_code=None,
                      seed: Optional[int] = None):
        """`iHQGPT.sampling_step` (hierarchical_ar.py:428-480).  `past` is an opaque token here: None starts a new
        batch (the reference asserts `past is None` at the first position, :494), anything else continues the batch
        whose KV cache the engine already holds.  Returns (code_top [B,1], code_bot [B,1,4], presents) where
        `presents` is that token."""
        B = sos.shape[0]
        eng = self._engine_for(use_fp16, B)
        S = self.max_seq_len
        if past is None:
            if codes_t is not None:
                raise AssertionError("first position: codes must be None when past is None")
            st = dict(pos=0, B=B, eng=eng, seed=fresh_seed() if seed is None else seed,   # one key per batch
                      codes_top=torch.zeros(B, S, dtype=torch.int64, device=self.device),
                      codes_bot=torch.zeros(B, S, 4, dtype=torch.int64, device=self.device))
            self._step_state = st
        else:
            st = self._step_state
            if st is None or st["B"] != B or st["eng"] is not eng:
                raise RuntimeError("sampling_step: `past` does not belong to the batch the engine holds")
            cnt = st["pos"]
            st["codes_top"][:, cnt - 1] = codes_t.reshape(B).to(self.device)
            st["codes_bot"][:, cnt - 1] = codes_b.reshape(B, 4).to(self.device)
            if pos_codes is not None and int(pos_codes.reshape(-1)[0]) != cnt - 1:
                raise ValueError(f"pos_codes {int(pos_codes.reshape(-1)[0])} != expected position {cnt - 1}")
        cnt = st["pos"]
        if cnt >= S:
            raise ValueError(f"position {cnt} beyond max_seq_len {S}")
        t_top, t_bot = _temps(softmax_temperature)
        sp = SamplingParams(top_k_top, top_p_top, top_k_bot, top_p_bot, t_top, t_bot,
                            seed=st["seed"] if seed is None else seed)
        given = None
        if given_top_code is not None:
            given = st["codes_top"].clone()
            given[:, cnt] = given_top_code.reshape(B).to(self.device)
        sos_dev = None
        if cnt == 0:
            sos_dev = sos.to(device=self.device, dtype=torch.float32).contiguous()
        eng.run(batch=B, seq_len=S, pos_begin=cnt, pos_end=cnt + 1, sampling=sp, sos=sos_dev, given_top=given,
                codes_top=st["codes_top"], codes_bot=st["codes_bot"])
        st["pos"] = cnt + 1
        code_top = st["codes_top"][:, cnt:cnt + 1].clone()
        code_bot = st["codes_bot"][:, cnt:cnt + 1, :].clone()
        return code_top, code_bot, ("hqgraft-kv", id(st), cnt)

    def build_sos(self, cond, num_candidates: int) -> Optional[torch.Tensor]:
        """Conditioning tensor for the engine: int64 [B] class ids, int64 [B, ctx_len_txt] text ids, or None."""
        if self.use_cls_cond:
            if isinstance(cond, int):
                if not 0 <= cond < self.n_classes:       # nn.Embedding would raise IndexError (sampling.py:186)
                    raise IndexError(f"class id {cond} out of range [0, {self.n_classes})")
                return torch.full((num_candidates,), cond, dtype=torch.int64, device=self.device)
            c = torch.as_tensor(cond, dtype=torch.int64).reshape(-1).to(self.device)
            if c.numel() and (int(c.min()) < 0 or int(c.max()) >= self.n_classes):
                raise IndexError(f"class ids out of range [0, {self.n_classes})")
            return c.repeat(num_candidates) if c.numel() == 1 else c
        if self.use_txt_cond:
            c = torch.as_tensor(cond, dtype=torch.int64).to(self.device).contiguous()
            if c.dim() != 2 or c.shape[1] != self.ctx_len_txt:
                raise ValueError(f"text condition must be int64 [B, {self.ctx_len_txt}], got {tuple(c.shape)}")
            if c.numel() and (int(c.min()) < 0 or int(c.max()) >= self.vocab_size_txt):
                raise IndexError(f"text token ids out of range [0, {self.vocab_size_txt})")
            return c
        return None


class ImageGPT2:
    """The object the scripts build from a config (hqvae/models/__init__.py:92-174): `.stage2` is the sampler.
    Stage 1 (HQ-VAE decoder) is outside this path; attach any module with the reference's
    `decode_code(code_t [B,8,8], code_b [B,16,16])` as `.stage1` to get pixels out of `sample()`.
    `stage1_precision` ("bf16" | "tf32") selects the format of the stage-1 decoder built with `with_stage1=True`."""

    def __init__(self, config, with_stage1: bool = False, stage1_max_batch: int = 16, stage1_precision: str = "bf16",
                 **engine_opts) -> None:
        from .stage1 import check_s1_precision
        check_s1_precision(stage1_precision)
        self.config = config
        self.stage1 = None
        if "multilevel-hq" in config.stage2.type:               # hqvae/models/__init__.py:138-145
            from .hqtransformer3 import HQTransformer
            engine_opts.pop("use_chain", None)
            self.stage2 = HQTransformer(**engine_kwargs(config), **engine_opts)
        else:
            self.stage2 = iHQGPT(**engine_kwargs(config), **engine_opts)
        if with_stage1:
            # the `decode_code` half of the HQ-VAE (hqvae/models/__init__.py:96-101 builds the whole generator)
            from .stage1 import HQVAEDecoder
            s1 = getattr(config, "stage1", None)
            if s1 is None:
                raise KeyError("with_stage1=True needs a `stage1` section in the config")
            self.stage1 = HQVAEDecoder.from_stage1_config(s1, max_batch=stage1_max_batch, device=self.stage2.device,
                                                          precision=stage1_precision)
        self.use_cls_cond = config.stage2.use_cls_cond
        self.use_txt_cond = config.stage2.use_txt_cond
        self.type = config.stage2.type

    @classmethod
    def from_config(cls, path: str, **engine_opts) -> "ImageGPT2":
        """`measure_throughput.load_model` (measure_throughput/__main__.py:25-31): config only, random-init weights."""
        model = cls(load_config(path), **engine_opts)
        model.stage2.init_weights(seed=0)
        if model.stage1 is not None:
            model.stage1.init_weights(seed=1)
        return model

    @classmethod
    def from_pretrained(cls, config_path: str, ckpt_path: str, **engine_opts) -> "ImageGPT2":
        """`sampling_hqmodel.load_model` (sampling_hqmodel.py:64-82): config + `ckpt['state_dict']`, strict."""
        model = cls(load_config(config_path), **engine_opts)
        sd = torch.load(ckpt_path, map_location="cpu")["state_dict"]
        model.load_state_dict(sd, strict=True)
        return model

    def load_state_dict(self, state_dict, strict: bool = True):
        """Accepts the full Lightning state_dict: 'stage2.*' keys feed the sampler engine; 'stage1.*' keys feed the stage-1
        decoder when one was built (`with_stage1=True`), else they are skipped."""
        s2 = {k[len("stage2."):]: v for k, v in state_dict.items() if k.startswith("stage2.")}
        if self.stage1 is not None and hasattr(self.stage1, "load_state_dict"):
            s1 = {k: v for k, v in state_dict.items() if k.startswith("stage1.")}
            if s1 or strict:
                self.stage1.load_state_dict(s1, strict=strict)
        other = [k for k in state_dict if not k.startswith(("stage1.", "stage2."))]
        if strict and other:
            raise KeyError(f"unexpected key(s) in state_dict: {other[:5]}")
        return self.stage2.load_state_dict(s2, strict=strict)

    def eval(self):
        self.stage2.eval()
        return self

    def to(self, device):
        self.stage2.to(device)
        return self

    @torch.no_grad()
    def sample(self, cls_idx: Optional[int] = None, top_k: int = 256, top_p: Optional[float] = None,
               softmax_temperature: float = 1.0, num_candidates: int = 16, device: str = "cuda:0",
               use_fp16: bool = True, is_tqdm: bool = True):
        """Keyword-compatible with `ImageGPT2.sample` (hqvae/models/__init__.py:207-215).  In the reference this
        entry only works for `type: top` models (SURVEY.md 3.4); here it routes HQ models to the hierarchical
        sampler.  Returns pixels when a stage-1 decoder is attached, else the code grids
        (codes_t [B,8,8], codes_b [B,16,16]) in the HQ-VAE layout."""
        from .sampling import codes_to_grids, sampling_ihqgpt
        codes_top, codes_bot = sampling_ihqgpt(self.stage2, cond=cls_idx, num_candidates=num_candidates,
                                               top_k_top=top_k, top_p_top=top_p, top_k_bot=top_k, top_p_bot=top_p,
                                               softmax_temperature=[softmax_temperature, softmax_temperature],
                                               use_fp16=use_fp16, is_tqdm=is_tqdm, max_seq_len=64)
        codes_t, codes_b = codes_to_grids(codes_top, codes_bot)
        if self.stage1 is None:
            return codes_t, codes_b
        return torch.clamp(self.stage1.decode_code(codes_t, codes_b) * 0.5 + 0.5, 0, 1)
