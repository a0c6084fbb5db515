"""Test-only fp16 rounding emulation for the oracles: the rounding points of their emulate="bf16" mode (GEMM weights,
GEMM-input activations, q / k / v and KV cache; fp32 everywhere else) with IEEE fp16 in place of bf16 - the rounding
points of the fp16 engine (HQ_PREC_F16).

Both oracles apply their 2-byte rounding through one module-level function, `_round_bf16`, which `round_params`, `sample`
(oracle/hq_oracle.py) and `_round_params3`, `sample` (oracle/hq3_oracle.py) look up when they are called.
`fp16_rounding()` replaces it by an fp16 rounding for the duration of a call and restores it afterwards, so the oracles
themselves stay exactly as they are.  tests/test_oracle_fp16.py checks that the substitution reaches every rounding point
(weights and activations) and that the bf16 emulation is unchanged afterwards."""
import contextlib

import torch

from oracle import hq3_oracle as O3
from oracle import hq_oracle as O


def round_fp16(t: torch.Tensor) -> torch.Tensor:
    return t.to(torch.float16).to(torch.float32)


@contextlib.contextmanager
def fp16_rounding():
    saved = O._round_bf16, O3._round_bf16
    O._round_bf16 = O3._round_bf16 = round_fp16
    try:
        yield
    finally:
        O._round_bf16, O3._round_bf16 = saved


def round_params(params):
    """The parameters as the fp16 engine stores them (GEMM weights and heads in fp16, the rest fp32)."""
    with fp16_rounding():
        return O.round_params(params, "bf16")


def round_params3(params):
    with fp16_rounding():
        return O3._round_params3(params, "bf16")


def step_logits(params, cfg, cond, codes_top, codes_bot):
    """O.step_logits with the fp16 engine's rounding points."""
    with fp16_rounding():
        return O.step_logits(params, cfg, cond, codes_top, codes_bot, emulate="bf16")


def sample3(params, cfg, cond, num_candidates, **kw):
    """O3.sample with the fp16 engine's rounding points."""
    with fp16_rounding():
        return O3.sample(params, cfg, cond, num_candidates, emulate="bf16", **kw)
