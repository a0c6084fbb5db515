"""Test-only TF32 rounding emulation for the stage-1 oracle: the rounding points of the tf32 decoder (HQ_PREC_TF32).

Every convolution input and every conv weight is rounded to TF32 with round-to-nearest, ties away from zero (what
`cvt.rna.tf32.f32` computes, the low 13 bits cleared); q / k / v, the attention core, the residual stream, GroupNorm and
biases stay fp32.

The oracle's emulate="bf16" mode rounds through one module-level function, `_rb`, which `decode_code` looks up when it is
called, and also rounds q / k / v in `_attnblock`.  `tf32_rounding()` replaces `_rb` by the TF32 rounding and `_attnblock`
by `_attnblock_fp32_qkv` (the oracle's AttnBlock without the q / k / v rounding) for the duration of a call and restores
both afterwards, so the oracle itself stays exactly as it is.  tests/test_stage1_tf32_cpu.py checks the rounding against
known answers and that the oracle is restored afterwards."""
import contextlib

import torch
from torch.nn import functional as F

from oracle import s1_oracle as S1


def round_tf32(t: torch.Tensor) -> torch.Tensor:
    """fp32 -> TF32 (10 explicit mantissa bits) rounded to nearest, ties away from zero; inf / NaN pass through."""
    u = t.float().contiguous().view(torch.int32)
    mag = ((u & 0x7FFFFFFF) + 0x1000) & 0x7FFFE000          # finite magnitudes are <= 0x7F7FFFFF: no int32 overflow
    r = mag | (u & torch.tensor(-0x80000000, dtype=torch.int32))
    return torch.where((u & 0x7F800000) == 0x7F800000, u, r).view(torch.float32)


def _attnblock_fp32_qkv(x, P, prefix, rnd, rw):                   # S1._attnblock with q / k / v left in fp32
    h = S1._gn(x, P, prefix + ".norm")
    q = S1._conv(h, P, prefix + ".q", 0, rnd, rw)
    k = S1._conv(h, P, prefix + ".k", 0, rnd, rw)
    v = S1._conv(h, P, prefix + ".v", 0, rnd, rw)
    b, c, hh, ww = q.shape
    q = q.reshape(b, c, hh * ww).permute(0, 2, 1)
    k = k.reshape(b, c, hh * ww)
    w_ = torch.softmax(torch.bmm(q, k) * (int(c) ** (-0.5)), dim=2)
    v = v.reshape(b, c, hh * ww)
    h = torch.bmm(v, w_.permute(0, 2, 1)).reshape(b, c, hh, ww)
    return x + S1._conv(h, P, prefix + ".proj_out", 0, rnd, rw)


@contextlib.contextmanager
def tf32_rounding():
    saved = S1._rb, S1._attnblock
    S1._rb, S1._attnblock = round_tf32, _attnblock_fp32_qkv
    try:
        yield
    finally:
        S1._rb, S1._attnblock = saved


def decode_code(P, cfg, code_t, code_b, accumulate=torch.float32):
    """S1.decode_code with the tf32 decoder's rounding points.  accumulate=torch.float64 computes everything between the
    rounding points in fp64 instead of fp32: two such emulations differ only in accumulation, and how far apart they end
    up is the floor for how close any fp32 implementation (the GPU's included) can come to this one - a value near a TF32
    rounding boundary rounds either way depending on summation order, and ~40 layers follow."""
    if accumulate == torch.float32:
        with tf32_rounding():
            return S1.decode_code(P, cfg, code_t, code_b, emulate="bf16")
    with tf32_rounding():
        S1._rb = lambda t: round_tf32(t).to(accumulate)
        out = S1.decode_code({k: v.to(accumulate) for k, v in P.items()}, cfg, code_t, code_b, emulate="bf16")
    return out.float()


def conv_fp64(A_nhwc: torch.Tensor, weight: torch.Tensor, bias: torch.Tensor, k: int, round_weight=round_tf32):
    """fp64 convolution of a padded NHWC operand [B, res+2, res+2, Cin] (as stored) with fp32 weights rounded as the
    decoder packs them (round_weight: TF32 by default), and the same of |A| * |W| (the scale of the fp32 accumulation
    error): both [B, Cout, res, res]."""
    a = A_nhwc[:, 1:-1, 1:-1, :].permute(0, 3, 1, 2).double()
    w = round_weight(weight).double()
    y = F.conv2d(a, w, bias.double(), padding=k // 2)
    s = F.conv2d(a.abs(), w.abs(), None, padding=k // 2)
    return y, s
