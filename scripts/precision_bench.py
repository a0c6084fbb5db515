"""The bf16 and fp16 engines side by side on the flagship workload (ImageNet L12, B = 256, 64 top positions, top-k / top-p
None, T = 1 - bench.py's default sampling):

    python scripts/precision_bench.py [--batch 256] [--rounds 4] [--steps 3] [--out DIR]

Both engines are built from the same config with the same seeded weights (`ImageGPT2.from_config`), and timed in
alternating rounds inside one process (round r: bf16 then fp16, or fp16 then bf16), each round `steps` full sampling
calls between CUDA events after one warm-up call per engine.  The card's name and power limit are read in the same run.
It also reports the teacher-forced logits drift of each engine against the fp32 engine on the same seeded inputs
(max-abs, mean-abs, greedy flips).  One JSON line goes to stdout (and to DIR/precision_bench.json with --out).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card_info(index: int) -> dict:
    info = {"name": torch.cuda.get_device_name(index), "power_limit_w": None, "max_sm_mhz": None}
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=power.limit,clocks.max.sm",
                              "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=30).stdout
        pl, mhz = [v.strip() for v in out.strip().split(",")[:2]]
        info["power_limit_w"], info["max_sm_mhz"] = float(pl), float(mhz)
    except Exception as e:                       # reported, not guessed
        info["query_error"] = str(e)
    return info


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--rounds", type=int, default=4)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import hqtransformer_b200 as H

    torch.set_grad_enabled(False)
    dev = torch.device("cuda", 0)
    B, S = args.batch, 64
    cfg = os.path.join(ROOT, "hqtransformer_b200", "configs", "imagenet_l12.yaml")
    models = {p: H.ImageGPT2.from_config(cfg, device=0, precision=p, max_batch=B).stage2 for p in ("bf16", "fp16", "fp32")}
    g = torch.Generator().manual_seed(1234)
    cond = torch.randint(0, models["bf16"].n_classes, (B,), generator=g).to(dev)
    kw = dict(top_k_top=None, top_k_bot=None, top_p_top=None, top_p_bot=None, softmax_temperature=[1.0, 1.0], use_fp16=True,
              max_seq_len=S, is_tqdm=False)

    def timed(p: str, seed: int) -> float:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(args.steps):
            H.sampling_ihqgpt(models[p], B, cond, seed=seed + i, **kw)
        e1.record()
        torch.cuda.synchronize()
        return B * args.steps / (e0.elapsed_time(e1) / 1000.0)

    for p in ("bf16", "fp16"):
        H.sampling_ihqgpt(models[p], B, cond, seed=0, **kw)
    torch.cuda.synchronize()
    rates = {"bf16": [], "fp16": []}
    for r in range(args.rounds):
        for p in (("bf16", "fp16") if r % 2 == 0 else ("fp16", "bf16")):
            rates[p].append(timed(p, 100 * r))

    # logits drift against the fp32 engine: 16 images, 8 teacher-forced positions, seeded codes
    gd = torch.Generator().manual_seed(7)
    Bd, Sd = 16, 8
    labels = torch.randint(0, models["bf16"].n_classes, (Bd,), generator=gd)
    ct = torch.randint(0, models["bf16"].vocab_size_top, (Bd, Sd), generator=gd)
    cb = torch.randint(0, models["bf16"].vocab_size_bot, (Bd, Sd, 4), generator=gd)
    ref = H.step_logits(models["fp32"], labels, ct, cb, use_fp16=False).double()
    drift = {}
    for p in ("bf16", "fp16"):
        lg = H.step_logits(models[p], labels, ct, cb, use_fp16=True).double()
        d = (lg - ref).abs()
        flips = (lg.argmax(-1) != ref.argmax(-1))
        drift[p] = {"max_abs": d.max().item(), "mean_abs": d.mean().item(), "greedy_flips": int(flips.sum()),
                    "greedy_decisions": flips.numel()}

    res = {"workload": f"imagenet_l12 B={B} S={S} top_k/top_p None T=1", "card": card_info(0),
           "images_per_s": {p: {"median": statistics.median(v), "min": min(v), "max": max(v), "rounds": v}
                            for p, v in rates.items()},
           "fp16_over_bf16": statistics.median(rates["fp16"]) / statistics.median(rates["bf16"]),
           "logits_drift_vs_fp32_engine": drift}
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "precision_bench.json"), "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
