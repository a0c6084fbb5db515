"""Stage-1 decode of sampled code grids on the GPU: the `decode_code` half of `SimRQGAN2Generator`
(hqvae/models/stage1/generator.py:312-367), batched, behind libhqgraft's hq_s1_* entry points.

The scripts call `model.stage1.decode_code(code_t [B,8,8], code_b [B,16,16])` one image at a time after sampling
(sampling_hqmodel.py:197, measure_throughput/__main__.py:108-111); `HQVAEDecoder.decode_code` keeps that signature and
return value (float pixels [B, 3, R, R], the decoder's raw output) for any batch.  Supported configuration: the shipped
HQ-VAE (`type: simrqgan2`, `decoding_type: concat`, `upsample: pixelshuffle`, use_init_downsample / use_mid_block / use_attn).
"""
from __future__ import annotations

import ctypes as C
import math
from collections import OrderedDict
from typing import Dict, Optional, Tuple, Union

import torch

from . import _lib
from ._lib import HQS1Config, check_s1

_TORCH2HQ = {torch.float32: _lib.HQ_F32, torch.bfloat16: _lib.HQ_BF16, torch.float16: _lib.HQ_F16}
# operand format of the convolutions: "bf16" (default), or "tf32" - the reference's own (decode_code runs in fp32 outside
# autocast and cuDNN runs its convolutions in TF32); see HQ_PREC_TF32 in include/hqgraft.h
S1_PRECISIONS = {"bf16": _lib.HQ_PREC_BF16, "tf32": _lib.HQ_PREC_TF32}


def check_s1_precision(precision: str) -> int:
    if precision not in S1_PRECISIONS:
        raise ValueError(f"stage-1 precision {precision!r}: one of {sorted(S1_PRECISIONS)}")
    return S1_PRECISIONS[precision]


class HQVAEDecoder:
    """`stage1` of an `ImageGPT2`: only what `decode_code` needs (codebooks, post_quant_conv_b, Decoder).
    precision: "bf16" (default) or "tf32" (the reference's format: TF32 convolutions, fp32 attention and residual stream)."""

    def __init__(self, *, embed_dim: int = 256, n_embed: int = 8192, z_channels: int = 256, resolution: int = 256,
                 ch: int = 128, ch_mult=(1, 2, 4, 4), num_res_blocks: int = 2, attn_resolutions=(16,), out_ch: int = 3,
                 max_batch: int = 16, device: Union[int, str, torch.device] = 0, precision: str = "bf16"):
        prec = check_s1_precision(precision)
        self.precision = precision
        self._lib = _lib.load()
        self._ctx = C.c_void_p()
        dev = torch.device(device) if not isinstance(device, int) else torch.device("cuda", device)
        if dev.type != "cuda":
            raise ValueError("hqtransformer_b200 runs on CUDA (sm_100a) devices only; there is no CPU path")
        self.device = torch.device("cuda", dev.index or 0)
        if len(attn_resolutions) != 1:
            raise NotImplementedError("exactly one attention resolution (the shipped configs use [16])")
        self.embed_dim, self.n_embed, self.z_channels, self.resolution = embed_dim, n_embed, z_channels, resolution
        self.ch, self.ch_mult, self.num_res_blocks, self.out_ch = ch, tuple(ch_mult), num_res_blocks, out_ch
        self.attn_resolution = int(attn_resolutions[0])
        self.latent_res = resolution // 2 ** len(self.ch_mult)
        self.max_batch = int(max_batch)
        mult = (C.c_int32 * 8)(*(list(self.ch_mult) + [0] * (8 - len(self.ch_mult))))
        cfg = HQS1Config(embed_dim=embed_dim, n_embed=n_embed, z_channels=z_channels, resolution=resolution, ch=ch,
                         ch_mult=mult, n_levels=len(self.ch_mult), num_res_blocks=num_res_blocks,
                         attn_resolution=self.attn_resolution, out_ch=out_ch, precision=prec)
        check_s1(self._lib.hq_s1_create(C.byref(cfg), self.device.index, self.max_batch, C.byref(self._ctx)), None,
                 self._lib, "hq_s1_create")

    @classmethod
    def from_stage1_config(cls, s1, **kw) -> "HQVAEDecoder":
        """From the `stage1` section of a reference YAML (namespace or dict); `kw` (max_batch, device, precision) pass through."""
        get = (lambda o, k, d=None: o.get(k, d)) if isinstance(s1, dict) else (lambda o, k, d=None: getattr(o, k, d))
        if get(s1, "type") not in (None, "simrqgan2"):
            raise NotImplementedError(f"stage1.type={get(s1, 'type')!r}: only 'simrqgan2' (2-level HQ-VAE) is implemented")
        hp, aux = get(s1, "hparams"), get(s1, "hparams_aux")
        if aux is not None and (get(aux, "decoding_type", "concat") != "concat" or get(aux, "upsample", "pixelshuffle") != "pixelshuffle"):
            raise NotImplementedError("only decoding_type 'concat' with upsample 'pixelshuffle' is implemented")
        for flag in ("use_init_downsample", "use_mid_block", "use_attn"):
            if not get(hp, flag, True):
                raise NotImplementedError(f"stage1.hparams.{flag}=False is not implemented")
        return cls(embed_dim=get(s1, "embed_dim"), n_embed=get(s1, "n_embed"), z_channels=get(hp, "z_channels"),
                   resolution=get(hp, "resolution"), ch=get(hp, "ch"), ch_mult=tuple(get(hp, "ch_mult")),
                   num_res_blocks=get(hp, "num_res_blocks"), attn_resolutions=tuple(get(hp, "attn_resolutions")),
                   out_ch=get(hp, "out_ch", 3), **kw)

    # ---- lifetime ----
    def close(self) -> None:
        if getattr(self, "_ctx", None) is not None and self._ctx.value:
            self._lib.hq_s1_destroy(self._ctx)
            self._ctx = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def device_bytes(self) -> int:
        return self._lib.hq_s1_device_bytes(self._ctx)

    @property
    def last_conv_flops(self) -> float:
        return self._lib.hq_s1_last_conv_flops(self._ctx)

    # ---- parameters ----
    def param_shapes(self) -> "OrderedDict[str, Tuple[int, ...]]":
        """The generator state_dict keys `decode_code` reads (generator.py:243-250, stage1/modules/layers.py:300-383)."""
        s: "OrderedDict[str, Tuple[int, ...]]" = OrderedDict()
        E = self.embed_dim

        def res(p, cin, cout):
            s[p + ".norm1.weight"] = (cin,); s[p + ".norm1.bias"] = (cin,)
            s[p + ".conv1.weight"] = (cout, cin, 3, 3); s[p + ".conv1.bias"] = (cout,)
            s[p + ".norm2.weight"] = (cout,); s[p + ".norm2.bias"] = (cout,)
            s[p + ".conv2.weight"] = (cout, cout, 3, 3); s[p + ".conv2.bias"] = (cout,)
            if cin != cout:
                s[p + ".nin_shortcut.weight"] = (cout, cin, 1, 1); s[p + ".nin_shortcut.bias"] = (cout,)

        def attn(p, c):
            s[p + ".norm.weight"] = (c,); s[p + ".norm.bias"] = (c,)
            for nm in ("q", "k", "v", "proj_out"):
                s[f"{p}.{nm}.weight"] = (c, c, 1, 1); s[f"{p}.{nm}.bias"] = (c,)

        s["quantize_t.embedding"] = (self.n_embed, 4 * E)
        s["quantize_b.embedding"] = (self.n_embed, E)
        s["post_quant_conv_b.weight"] = (self.z_channels, 2 * E, 1, 1)
        s["post_quant_conv_b.bias"] = (self.z_channels,)
        top = self.ch * self.ch_mult[-1]
        s["decoder.conv_in.weight"] = (top, self.z_channels, 3, 3)
        s["decoder.conv_in.bias"] = (top,)
        res("decoder.mid.block_1", top, top)
        attn("decoder.mid.attn_1", top)
        res("decoder.mid.block_2", top, top)
        block_in, r = top, self.latent_res
        for lvl in reversed(range(len(self.ch_mult))):
            block_out = self.ch * self.ch_mult[lvl]
            for j in range(self.num_res_blocks + 1):
                res(f"decoder.up.{lvl}.block.{j}", block_in, block_out)
                block_in = block_out
                if r == self.attn_resolution:
                    attn(f"decoder.up.{lvl}.attn.{j}", block_in)
            s[f"decoder.up.{lvl}.upsample.conv.weight"] = (block_in, block_in, 3, 3)
            s[f"decoder.up.{lvl}.upsample.conv.bias"] = (block_in,)
            r *= 2
        s["decoder.norm_out.weight"] = (block_in,); s["decoder.norm_out.bias"] = (block_in,)
        s["decoder.conv_out.weight"] = (self.out_ch, block_in, 3, 3); s["decoder.conv_out.bias"] = (self.out_ch,)
        return s

    def load_param(self, name: str, t: torch.Tensor) -> None:
        t = t.detach()
        if t.dtype not in _TORCH2HQ:
            t = t.float()
        t = t.contiguous()
        if t.is_cuda and t.device != self.device:
            t = t.to(self.device)
        shape = (C.c_int64 * t.dim())(*t.shape)
        check_s1(self._lib.hq_s1_load_param(self._ctx, name.encode(), t.data_ptr(), _TORCH2HQ[t.dtype], shape, t.dim(),
                                            1 if t.is_cuda else 0), self._ctx, self._lib, f"hq_s1_load_param({name})")

    def load_state_dict(self, sd: Dict[str, torch.Tensor], strict: bool = True):
        """Keys of the reference generator (optionally prefixed 'stage1.').  The encoder / quant_conv_b / EMA statistics of a
        full checkpoint are not part of decode_code and are skipped; every key decode_code reads must be present."""
        want = self.param_shapes()
        for k, v in sd.items():
            k = k[len("stage1."):] if k.startswith("stage1.") else k
            if k in want:
                self.load_param(k, v)
            elif strict and not k.startswith(("encoder.", "quant_conv_b.", "quantize_t.", "quantize_b.", "loss.")):
                raise _lib.HQError(f"unexpected key in stage-1 state_dict: {k!r}")
        if strict:
            check_s1(self._lib.hq_s1_params_complete(self._ctx), self._ctx, self._lib, "load_state_dict")

    @torch.no_grad()
    def init_weights(self, seed: int = 0) -> None:
        """Synthetic weights (conv ~ N(0, 1/fan_in), GroupNorm (1, 0), codebooks ~ N(0, 1)): what a throughput run without a
        checkpoint decodes with (measure_throughput/__main__.py:25-31 builds the model from the config alone)."""
        g = torch.Generator(device=self.device).manual_seed(seed)
        for name, shape in self.param_shapes().items():
            leaf = name.split(".")[-1]
            if "norm" in name:
                t = torch.ones(shape, device=self.device) if leaf == "weight" else torch.zeros(shape, device=self.device)
            elif leaf == "bias":
                t = torch.zeros(shape, device=self.device)
            elif leaf == "embedding":
                t = torch.randn(shape, generator=g, device=self.device)
            else:
                t = torch.randn(shape, generator=g, device=self.device) / math.sqrt(shape[1] * shape[2] * shape[3])
            self.load_param(name, t)
            del t

    def eval(self):
        return self

    # ---- the reference call ----
    @torch.no_grad()
    def decode_code(self, code_t: torch.Tensor, code_b: torch.Tensor) -> torch.Tensor:
        """generator.py:323-367 with both grids: code_t int64 [B, h, w], code_b int64 [B, 2h, 2w] -> float32 [B, out_ch, R, R].
        Batches above `max_batch` are decoded in chunks."""
        if code_t is None or code_b is None:
            raise NotImplementedError("decode_code needs both grids (top-only / bottom-only decoding is not implemented)")
        h = self.latent_res // 2
        ct = code_t.to(device=self.device, dtype=torch.int64).contiguous()
        cb = code_b.to(device=self.device, dtype=torch.int64).contiguous()
        B = ct.shape[0]
        if tuple(ct.shape) != (B, h, h) or tuple(cb.shape) != (B, 2 * h, 2 * h):
            raise ValueError(f"expected code_t [B,{h},{h}] and code_b [B,{2 * h},{2 * h}], got {tuple(ct.shape)} / {tuple(cb.shape)}")
        if B and (int(ct.min()) < 0 or int(ct.max()) >= self.n_embed or int(cb.min()) < 0 or int(cb.max()) >= self.n_embed):
            raise IndexError(f"code indices out of range [0, {self.n_embed})")
        out = torch.empty(B, self.out_ch, self.resolution, self.resolution, dtype=torch.float32, device=self.device)
        st = torch.cuda.current_stream(self.device).cuda_stream
        for lo in range(0, B, self.max_batch):
            hi = min(B, lo + self.max_batch)
            check_s1(self._lib.hq_s1_decode_codes(self._ctx, ct[lo:hi].data_ptr(), cb[lo:hi].data_ptr(), out[lo:hi].data_ptr(),
                                                  hi - lo, C.c_void_p(st)), self._ctx, self._lib, "hq_s1_decode_codes")
        return out


def debug_s1_conv(A: torch.Tensor, weight: torch.Tensor, bias: torch.Tensor, out: torch.Tensor, mode: int, *,
                  resid: Optional[torch.Tensor] = None, tile: int = 0) -> None:
    """One decoder convolution through hq_debug_s1_conv (weight packing, tile planner and conv kernel of the decoder),
    in place, synchronous.  A: padded NHWC [B, res+2, res+2, Cin], bf16 (precision bf16) or fp32 (tf32: already rounded);
    weight fp32 [Cout, Cin, k, k]; bias fp32 [Cout].  mode 0: out fp32 [B, res+2, res+2, Cout] (+= resid, which may be out);
    1: out in A's dtype, same layout; 2: out fp32 [B, Cout, res, res].  tile 0: the planner's width."""
    lib = _lib.load()
    prec = {torch.bfloat16: _lib.HQ_PREC_BF16, torch.float32: _lib.HQ_PREC_TF32}[A.dtype]
    B, Hp, _, Cin = A.shape
    Cout, _, k, _ = weight.shape
    for t in (A, weight, bias, out) + ((resid,) if resid is not None else ()):
        assert t.is_cuda and t.is_contiguous() and t.device == A.device
    assert weight.dtype == bias.dtype == torch.float32 and out.dtype == (A.dtype if mode == 1 else torch.float32)
    with torch.cuda.device(A.device):
        st = torch.cuda.current_stream(A.device).cuda_stream
        rc = lib.hq_debug_s1_conv(prec, A.data_ptr(), weight.data_ptr(), bias.data_ptr(), B, Hp - 2, Cin, Cout, k, mode,
                                  tile, resid.data_ptr() if resid is not None else None, out.data_ptr(), C.c_void_p(st))
        check_s1(rc, None, lib, "hq_debug_s1_conv")
