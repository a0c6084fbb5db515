"""Full-context sampling and 512 x 512 decode on one GPU: ImageNet L12 (random init), bf16 engine, top-k / top-p None,
all 256 top positions, and the stage-1 decoder on 16 x 16 / 32 x 32 grids.

    python scripts/long_context_bench.py [--batch 256] [--reps 3] [--out profiles/long_context_B256.json]

Reports images/s and ms per call of the 256-position sampler, the device time of single positions t = 64 / 128 / 192 /
255 (hq_trace_run), the decode attention's achieved bandwidth there (2 (t + 1) D 2 bytes of K / V per image and layer over
the kernel's device time), and stage-1 ms per 512 x 512 image at B = 8 in bf16 and tf32 with the AttnBlock share
(torch.profiler).  Card name and power limit are read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

from precision_bench import card_info  # noqa: E402

HBM_DATASHEET = 7.7e12      # B/s, HGX B200 data sheet, one GPU


def sampler(B: int, reps: int) -> dict:
    import hqtransformer_b200 as H
    from hqtransformer_b200.engine import SamplingParams
    model = H.ImageGPT2.from_config(os.path.join(ROOT, "hqtransformer_b200", "configs", "imagenet_l12.yaml"), device=0,
                                    precision="bf16", max_batch=B, max_seq_len=256)
    s2 = model.stage2
    cond = torch.randint(0, 1000, (B,), device="cuda", generator=torch.Generator(device="cuda").manual_seed(0))
    kw = dict(top_k_top=None, top_p_top=None, top_k_bot=None, top_p_bot=None, softmax_temperature=[1.0, 1.0],
              is_tqdm=False, max_seq_len=256)
    ct, cb = H.sampling_ihqgpt(s2, B, cond, **kw)         # warm-up: graphs captured, cache filled
    torch.cuda.synchronize()
    times = []
    for _ in range(reps):
        t0 = time.perf_counter()
        ct, cb = H.sampling_ihqgpt(s2, B, cond, **kw)
        torch.cuda.synchronize()
        times.append(time.perf_counter() - t0)
    ms = 1e3 * min(times)
    eng = s2.engine("bf16")
    D, L = s2.embed_dim, s2.n_layers
    per_pos = {}
    for t in (64, 128, 192, 255):
        for _ in range(2):      # second pass is the one kept (warm)
            tl = eng.trace_run(batch=B, seq_len=256, pos_begin=t, pos_end=t + 1, sampling=SamplingParams(), cond=cond,
                               codes_top=ct, codes_bot=cb)
        span = (max(e for _, _, e in tl) - min(s for _, s, _ in tl)) * 1e-6
        att = [(tag, e - s) for tag, s, e in tl if tag.startswith("attention_decode:t")]
        att_ns = sum(d for _, d in att)
        keys = int(att[0][0].split(":t")[1].split(":")[0]) if att else 0
        kv_bytes = 2.0 * keys * D * 2 * B * len(att)
        per_pos[str(t)] = {"position_ms": span, "attention_launches": len(att), "attention_ms": att_ns * 1e-6, "keys": keys,
                           "attention_tb_per_s": kv_bytes / (att_ns * 1e-9) / 1e12 if att_ns else None,
                           "attention_hbm_fraction_of_datasheet": kv_bytes / (att_ns * 1e-9) / HBM_DATASHEET if att_ns else None}
    return {"batch": B, "layers": L, "embed_dim": D, "positions": 256, "ms_per_call": ms, "images_per_s": B / (ms * 1e-3),
            "all_reps_ms": [1e3 * x for x in times], "per_position": per_pos}


def stage1(precision: str, B: int = 8, reps: int = 5) -> dict:
    import hqtransformer_b200 as H
    from torch.profiler import ProfilerActivity, profile
    conf = H.load_config(os.path.join(ROOT, "hqtransformer_b200", "configs", "imagenet_l12.yaml"))
    dec = H.HQVAEDecoder.from_stage1_config(conf.stage1, max_batch=B, device=0, precision=precision)
    dec.init_weights(seed=1)
    g = torch.Generator().manual_seed(0)
    ct = torch.randint(0, dec.n_embed, (B, 16, 16), generator=g).cuda()
    cb = torch.randint(0, dec.n_embed, (B, 32, 32), generator=g).cuda()
    dec.decode_code(ct, cb)
    torch.cuda.synchronize()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    ev[0].record()
    for _ in range(reps):
        dec.decode_code(ct, cb)
    ev[1].record()
    torch.cuda.synchronize()
    ms = ev[0].elapsed_time(ev[1]) / reps
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        dec.decode_code(ct, cb)
        torch.cuda.synchronize()
    tot = att = 0.0
    for e in prof.key_averages():
        us = e.device_time_total if hasattr(e, "device_time_total") else e.cuda_time_total
        tot += us
        if "s1_attn" in e.key:
            att += us
    return {"precision": precision, "batch": B, "pixels": 512, "ms_per_image": ms / B,
            "attnblock_core_share": att / tot if tot else None}


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    res = {"card": card_info(0), "sampler_bf16": sampler(a.batch, a.reps),
           "stage1": [stage1("bf16"), stage1("tf32")]}
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
