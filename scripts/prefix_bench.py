"""Image completion on the flagship model (ImageNet L12, random init, bf16 engine, B = 256, 64 top positions, top-k / top-p
None, T = 1): the prefix pass against the forced loop.

    python scripts/prefix_bench.py [--batch 256] [--prefix 0,16,32,48] [--rounds 4] [--steps 3] [--out DIR]

For every prefix length P the same completion runs two ways, timed in alternating rounds (CUDA events around `steps` calls,
after one warm-up call of each):
  prefill  `sampling_ihqgpt(prefix_code_top=, prefix_code_bot=)`: one causal pass over the prefix, then positions P..63;
  forced   the loop over positions 0..P-1 with given_top + given_bot (every depth pass, head and draw thrown away), then a
           second call continuing at pos_begin = P - what the C ABI offered before.
The prefix is the first P positions of a grid the engine sampled with another seed.  Both paths use the same seed, so they
draw from the same Philox counters; the share of codes at positions >= P that agree is reported (they differ only where
the bf16 cache of the two paths differs in its last bits and that moves a draw).  Kernel times come from torch.profiler
(CUDA activity, after the timed rounds): the prefix attention launches inside one prefill call per P, and the kernel alone
(hq_debug_attention_prefix) at the prefix lengths used and at the text prefill's 64 queries, next to the per-(query, head)
warp kernel the text prefill runs.  The card's name and power limit are read in the same run.
One JSON line goes to stdout (and DIR/prefix_bench.json with --out).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

from precision_bench import card_info  # noqa: E402


def profiled_kernels(fn, substr: str):
    """(total device microseconds, launches) of the CUDA kernels whose name contains `substr` while fn() runs."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    us, n = 0.0, 0
    for evt in prof.key_averages():
        if substr in evt.key:
            us += getattr(evt, "device_time_total", None) or getattr(evt, "cuda_time_total", 0.0)
            n += evt.count
    return us, n


def kernel_us(E, B: int, n_q: int, heads: int, variant: int, iters: int = 20) -> float:
    """Mean device time of one prefix-attention launch (variant 0: attention_prefix_kernel, 1: attention_kernel)."""
    D = heads * 64
    g = torch.Generator(device="cuda").manual_seed(n_q)
    q = torch.randn(B, n_q, D, generator=g, device="cuda").bfloat16()
    K = torch.randn(B, n_q, D, generator=g, device="cuda").bfloat16()
    V = torch.randn(B, n_q, D, generator=g, device="cuda").bfloat16()
    E.debug_attention_prefix(q, K, V, variant=variant)      # warm-up
    name = "attention_prefix_kernel" if variant == 0 else "attention_kernel"

    def run():
        for _ in range(iters):
            E.debug_attention_prefix(q, K, V, variant=variant)
    us, n = profiled_kernels(run, name)
    return us / max(n, 1)


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--prefix", default="0,16,32,48")
    ap.add_argument("--rounds", type=int, default=4)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import hqtransformer_b200 as H
    from hqtransformer_b200 import engine as E

    torch.set_grad_enabled(False)
    dev = torch.device("cuda", 0)
    B, S = args.batch, 64
    cfg = os.path.join(ROOT, "hqtransformer_b200", "configs", "imagenet_l12.yaml")
    model = H.ImageGPT2.from_config(cfg, device=0, precision="bf16", max_batch=B).stage2
    eng = model.engine("bf16")
    g = torch.Generator().manual_seed(1234)
    cond = torch.randint(0, model.n_classes, (B,), generator=g).to(dev)
    kw = dict(top_k_top=None, top_k_bot=None, top_p_top=None, top_p_bot=None, softmax_temperature=[1.0, 1.0], use_fp16=True,
              max_seq_len=S, is_tqdm=False)
    src_t, src_b = H.sampling_ihqgpt(model, B, cond, seed=99, **kw)      # the grids whose prefixes are completed
    sp = lambda seed: E.SamplingParams(seed=seed)  # noqa: E731   (top-k / top-p None, T = 1, as kw)

    def prefill(P: int, seed: int):
        if P == 0:
            return H.sampling_ihqgpt(model, B, cond, seed=seed, **kw)
        return H.sampling_ihqgpt(model, B, cond, seed=seed, prefix_code_top=src_t[:, :P], prefix_code_bot=src_b[:, :P],
                                 shared_prefix=False, **kw)

    def forced(P: int, seed: int):
        ct, cb = src_t.clone(), src_b.clone()
        if P == 0:
            return H.sampling_ihqgpt(model, B, cond, seed=seed, **kw)
        eng.run(batch=B, seq_len=S, pos_begin=0, pos_end=P, sampling=sp(seed), cond=cond, given_top=src_t, given_bot=src_b,
                codes_top=ct, codes_bot=cb)
        eng.run(batch=B, seq_len=S, pos_begin=P, pos_end=S, sampling=sp(seed), cond=cond, codes_top=ct, codes_bot=cb)
        return ct, cb

    def timed(fn, P: int, seed: int) -> float:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(args.steps):
            fn(P, seed + i)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / args.steps

    prefixes = [int(v) for v in args.prefix.split(",")]
    out = {}
    for P in prefixes:
        a, b = prefill(P, 5), forced(P, 5)
        torch.cuda.synchronize()
        agree_t = float((a[0][:, P:] == b[0][:, P:]).float().mean())
        agree_b = float((a[1][:, P:] == b[1][:, P:]).float().mean())
        kept = bool(torch.equal(a[0][:, :P], src_t[:, :P]) and torch.equal(a[1][:, :P], src_b[:, :P]))
        ms = {"prefill": [], "forced": []}
        for r in range(args.rounds):
            for name in (("prefill", "forced") if r % 2 == 0 else ("forced", "prefill")):
                ms[name].append(timed(prefill if name == "prefill" else forced, P, 1000 * r))
        med = {k: statistics.median(v) for k, v in ms.items()}
        out[str(P)] = {"ms_per_call": {k: {"median": med[k], "min": min(v), "max": max(v), "rounds": v} for k, v in ms.items()},
                       "forced_over_prefill": med["forced"] / med["prefill"],
                       "agree_top_at_ge_P": agree_t, "agree_bot_at_ge_P": agree_b, "prefix_returned_unchanged": kept}

    for P in prefixes:
        if P > 0:
            prefill(P, 5)
            us, n = profiled_kernels(lambda: prefill(P, 5), "attention_prefix_kernel")
            out[str(P)]["prefix_attention_in_call"] = {"us_total": us, "launches": n}
    heads = model.n_heads
    kern = {}
    for n_q in sorted({p for p in prefixes if p > 0} | {64}):
        kern[str(n_q)] = {"prefix_kernel_us": kernel_us(E, B, n_q, heads, 0), "per_query_warp_kernel_us": kernel_us(E, B, n_q, heads, 1)}
    res = {"workload": f"imagenet_l12 random init, bf16, B={B} S={S} top_k/top_p None T=1", "card": card_info(0),
           "by_prefix_len": out, "attention_kernel_alone_B%d_heads%d" % (B, heads): kern}
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "prefix_bench.json"), "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
