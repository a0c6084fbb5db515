"""CPU: the TF32 rounding emulation of the stage-1 oracle (tests/tf32_emulation.py, the rounding points of the tf32
decoder) and the host side of precision="tf32"."""
import ctypes
import os
import re

import pytest
import torch

from oracle import s1_oracle as S1
from tests import tf32_emulation as T
from tests.helpers import load_golden

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _f(bits):
    return torch.tensor([bits], dtype=torch.int32).view(torch.float32)


def _bits(t):
    return t.contiguous().view(torch.int32)


def test_round_tf32_known_answers():
    one = 0x3F800000
    # exactly half a TF32 ulp (2^-11 at 1.0) rounds away from zero, on both signs
    assert _bits(T.round_tf32(_f(one + 0x1000))).item() == one + 0x2000
    assert _bits(T.round_tf32(-_f(one + 0x1000))).item() == _bits(-_f(one + 0x2000)).item()
    # ties go away whatever the parity of the TF32 mantissa (nearest-even would round 0x5000 down to 0x4000)
    assert _bits(T.round_tf32(_f(one + 0x3000))).item() == one + 0x4000
    assert _bits(T.round_tf32(_f(one + 0x5000))).item() == one + 0x6000
    # below / above half an ulp
    assert _bits(T.round_tf32(_f(one + 0x0FFF))).item() == one
    assert _bits(T.round_tf32(_f(one + 0x1001))).item() == one + 0x2000
    # carry into the exponent: 2 - 2^-24 -> 2
    assert T.round_tf32(_f(0x3FFFFFFF)).item() == 2.0
    # inf / nan / zeros pass through
    x = torch.tensor([float("inf"), float("-inf"), 0.0, -0.0])
    assert torch.equal(_bits(T.round_tf32(x)), _bits(x))
    assert torch.isnan(T.round_tf32(torch.tensor([float("nan")]))).all()


def test_round_tf32_keeps_representable_values_and_clears_low_bits():
    g = torch.Generator().manual_seed(0)
    x = torch.randn(100000, generator=g) * torch.exp(8 * torch.randn(100000, generator=g))
    r = T.round_tf32(x)
    assert (_bits(r) & 0x1FFF).eq(0).all()
    assert torch.equal(T.round_tf32(r), r)
    # within half an ulp (2^-11 relative)
    assert ((r - x).abs() <= x.abs() * 2.0 ** -11).all()
    # agrees with round-to-nearest-even except on exact ties
    tie = (_bits(x) & 0x1FFF) == 0x1000
    rne = (_bits(x) + 0x0FFF + ((_bits(x) >> 13) & 1)) & ~0x1FFF
    assert torch.equal(_bits(r)[~tie], rne[~tie])


def test_tf32_emulation_rounds_conv_inputs_not_qkv_and_restores_the_oracle():
    cfg = S1.TINY_S1
    P = S1.make_params(cfg, seed=3)
    g = torch.Generator().manual_seed(1)
    h = cfg.latent_res // 2
    ct = torch.randint(0, cfg.n_embed, (2, h, h), generator=g)
    cb = torch.randint(0, cfg.n_embed, (2, 2 * h, 2 * h), generator=g)
    rb, attn = S1._rb, S1._attnblock
    seen = []

    def spy(t):
        seen.append(t)
        return T.round_tf32(t)
    with T.tf32_rounding():
        S1._rb = spy
        tf = S1.decode_code(P, cfg, ct, cb, emulate="bf16")
    assert S1._rb is rb and S1._attnblock is attn
    n_conv = sum(1 for k in P if k.endswith(".weight") and P[k].dim() == 4)
    assert len(seen) == 2 * n_conv                     # one input + one weight per convolution, nothing else
    fp = S1.decode_code(P, cfg, ct, cb)
    bf = S1.decode_code(P, cfg, ct, cb, emulate="bf16")
    e_tf, e_bf = (tf - fp).abs(), (bf - fp).abs()
    assert 0 < float(e_tf.max()) < 1e-2 and float(e_tf.mean()) < 0.3 * float(e_bf.mean())


def test_oracle_unchanged_after_tf32_emulation_reproduces_golden():
    g, meta = load_golden("s1_tiny_decode.npz")
    cfg = S1.S1Config.from_dict(meta["config"])
    P = S1.make_params(cfg, seed=meta["seed"])
    ct, cb = torch.from_numpy(g["code_t"]), torch.from_numpy(g["code_b"])
    T.decode_code(P, cfg, ct[:1], cb[:1])
    got = S1.decode_code(P, cfg, ct, cb)
    want = torch.from_numpy(g["pixels"])
    assert float((got - want).abs().max()) <= 1e-4


def test_bad_stage1_precision_strings_raise_before_device_work():
    import hqtransformer_b200 as H
    from hqtransformer_b200 import measure_throughput as M
    for bad in ("fp16", "fp32", "TF32", ""):
        with pytest.raises(ValueError):
            H.HQVAEDecoder(precision=bad)
        with pytest.raises(ValueError):
            H.ImageGPT2(None, with_stage1=True, stage1_precision=bad)
    args = M.parse_cli(["model_path=x.yaml", "stage1_precision=tf32"])
    assert args.stage1_precision == "tf32"


def test_header_and_binding_agree_on_abi_9_and_the_stage1_config():
    from hqtransformer_b200 import _lib
    header = open(os.path.join(ROOT, "include", "hqgraft.h")).read()
    assert _lib.ABI_VERSION == 9 and int(re.search(r"#define HQ_ABI_VERSION (\d+)", header).group(1)) == 9
    assert _lib.load().hq_abi_version() == 9
    assert re.search(r"HQ_PREC_TF32 = 3", header) and _lib.HQ_PREC_TF32 == 3
    body = re.search(r"typedef struct hq_s1_config \{(.*?)\} hq_s1_config;", header, re.S).group(1)
    fields = re.findall(r"int32_t (\w+)(?:\[(\d+)\])?;", body)
    assert [f for f, _ in fields] == [f for f, _ in _lib.HQS1Config._fields_]
    assert fields[-1][0] == "precision"
    assert ctypes.sizeof(_lib.HQS1Config) == 4 * sum(int(n or 1) for _, n in fields) == 18 * 4
    assert "hq_debug_s1_conv" in _lib.PROTOTYPES and "hq_debug_s1_conv" in header


def test_tf32_emulation_with_fp64_accumulation_restores_the_oracle():
    cfg = S1.TINY_S1
    P = S1.make_params(cfg, seed=3)
    h = cfg.latent_res // 2
    ct, cb = torch.zeros(1, h, h, dtype=torch.long), torch.ones(1, 2 * h, 2 * h, dtype=torch.long)
    rb, attn = S1._rb, S1._attnblock
    e64 = T.decode_code(P, cfg, ct, cb, accumulate=torch.float64)
    assert S1._rb is rb and S1._attnblock is attn
    assert e64.dtype == torch.float32 and float((e64 - T.decode_code(P, cfg, ct, cb)).abs().max()) < 1e-2
