"""CPU: the fp16 rounding emulation of the oracles (tests/fp16_emulation.py, the rounding points of the fp16 engine) and
the host side of precision="fp16"."""
import os
import re

import pytest

import torch

from oracle import hq3_oracle as O3
from oracle import hq_oracle as O
from tests import fp16_emulation as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_fp16_params_round_gemm_weights_only_and_bf16_is_restored():
    cfg = O.TINY
    P = O.make_params(cfg, seed=1, init="rich")
    R = F.round_params(P)
    assert list(R) == list(P)
    for k, v in P.items():
        gemm = k.endswith(O._GEMM_WEIGHT_LEAVES) or k in ("head_top.weight", "head_bot.weight")
        want = v.half().float() if gemm else v
        assert torch.equal(R[k], want), k
        assert R[k].dtype == torch.float32
    # the substitution is undone: the oracles' own bf16 emulation is what it was
    assert O._round_bf16 is not F.round_fp16 and O3._round_bf16 is not F.round_fp16
    Rb = O.round_params(P, "bf16")
    assert torch.equal(Rb["head_top.weight"], P["head_top.weight"].to(torch.bfloat16).float())


def test_fp16_emulation_sits_between_fp32_and_bf16():
    """Teacher-forced logits: the fp16 emulation is closer to fp32 than the bf16 emulation (3 more mantissa bits at the
    same rounding points) and does round.  With only the weights rounded to fp16 (activations left in fp32) the result
    differs from the full emulation: the activation rounding points are reached too."""
    cfg = O.SMALL
    P = O.make_params(cfg, seed=3, init="rich")
    g = torch.Generator().manual_seed(0)
    B, S = 3, 3
    labels = torch.randint(0, cfg.n_classes, (B,), generator=g)
    ct = torch.randint(0, cfg.vocab_top, (B, S), generator=g)
    cb = torch.randint(0, cfg.vocab_bot, (B, S, 4), generator=g)
    ref = O.step_logits(P, cfg, labels, ct, cb)
    l16 = F.step_logits(P, cfg, labels, ct, cb)
    e16 = (l16 - ref).abs().max().item()
    eb = (O.step_logits(P, cfg, labels, ct, cb, emulate="bf16") - ref).abs().max().item()
    weights_only = O.step_logits(F.round_params(P), cfg, labels, ct, cb)
    print(f"oracle max-abs vs fp32: fp16 emulation {e16:.3e}, bf16 emulation {eb:.3e}")
    assert 0.0 < e16 < 0.5 * eb
    assert not torch.equal(weights_only, l16)


def test_level3_oracle_fp16_emulation():
    cfg = O3.TINY3
    P = O3.make_params(cfg, seed=7)
    B, S = 2, 2
    g = torch.Generator().manual_seed(1)
    labels = torch.randint(0, cfg.n_classes, (B,), generator=g)
    given = torch.stack([torch.randint(0, cfg.vocab_sizes[0 if j == 0 else (1 if j < 5 else 2)], (B, S), generator=g)
                         for j in range(21)], dim=-1)
    _, ref = O3.sample(P, cfg, labels, B, max_seq_len=S, given=given, return_logits=True)
    _, l16 = F.sample3(P, cfg, labels, B, max_seq_len=S, given=given, return_logits=True)
    _, lbf = O3.sample(P, cfg, labels, B, max_seq_len=S, given=given, return_logits=True, emulate="bf16")
    e16, eb = (l16 - ref).abs().max().item(), (lbf - ref).abs().max().item()
    assert 0.0 < e16 < 0.5 * eb, (e16, eb)
    R = F.round_params3(P)
    for k in P:
        if k.startswith("head_levels."):
            assert torch.equal(R[k], P[k].half().float())


def test_fp16_precision_is_in_the_abi_and_the_host_layer():
    from hqtransformer_b200 import _lib
    from hqtransformer_b200.measure_throughput import parse_cli
    header = open(os.path.join(ROOT, "include", "hqgraft.h")).read()
    enum = re.search(r"enum hq_precision \{([^}]*)\}", header).group(1)
    assert "HQ_PREC_F16 = 2" in enum and _lib.HQ_PREC_F16 == 2 and _lib.HQ_PREC["fp16"] == 2
    assert _lib.HQ_PREC == {"bf16": 0, "fp32": 1, "fp16": 2}
    assert parse_cli(["model_path=x.yaml"]).precision == "bf16"
    assert parse_cli(["model_path=x.yaml", "precision=fp16"]).precision == "fp16"


def test_unknown_precision_is_rejected_before_the_library_is_touched():
    from hqtransformer_b200.engine import Engine
    with pytest.raises(ValueError, match="precision"):
        Engine(embed_dim=64, n_heads=1, n_layers=1, n_layers_depth=1, vocab_top=64, vocab_bot=64, precision="fp8")
