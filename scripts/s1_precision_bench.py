"""Stage-1 decode in its two formats and PyTorch's: the shipped HQ-VAE decoder (256 x 256, random-init weights) on random
grids at batch B (default 32).

    python scripts/s1_precision_bench.py [--batch 32] [--rounds 5] [--iters 5]

Arms, timed in alternating rounds so that clock and neighbour load drift hit all of them alike:
  bf16     HQVAEDecoder(precision="bf16")
  tf32     HQVAEDecoder(precision="tf32")
  pytorch  the stage-1 oracle's ops (oracle/s1_oracle.decode_code: the reference's layer sequence, functional) run by
           PyTorch on the GPU, batched, under its defaults: cuDNN convolutions in TF32, bmm in fp32 - what the reference's
           decode_code computes there
Each arm's time is CUDA events around `iters` back-to-back decodes of the same batch (the activations of one decode,
~1 GB at B = 32, exceed the 126 MB L2).  Prints one JSON line per arm and round, then a summary line: median ms per image,
min-max over rounds, conv TFLOP/s (2 x MACs of the convolutions, interior pixels, over the whole decode time) against
the data-sheet dense rate of the format (TF32 1 125, BF16 2 250 TFLOP/s per B200), and the GPU's name and power limit
read in the same run."""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import hqtransformer_b200 as H  # noqa: E402
from oracle import s1_oracle as S1  # noqa: E402

DATASHEET_TFLOPS = {"bf16": 2250.0, "tf32": 1125.0, "pytorch": 1125.0}


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    line = q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else ""
    name, power, clock = ([s.strip() for s in line.split(",")] + ["?", "?", "?"])[:3]
    return {"gpu": name or torch.cuda.get_device_name(0), "power_limit": power, "max_sm_clock": clock}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=32)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--iters", type=int, default=5)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("s1_precision_bench.py measures on a CUDA GPU; none is visible")
    B = a.batch
    dev = torch.device("cuda", 0)
    info = gpu_info()
    g = torch.Generator(device=dev).manual_seed(0)
    ct = torch.randint(0, 8192, (B, 8, 8), device=dev, generator=g)
    cb = torch.randint(0, 8192, (B, 16, 16), device=dev, generator=g)
    decs = {}
    for prec in ("bf16", "tf32"):
        decs[prec] = H.HQVAEDecoder(max_batch=B, precision=prec)
        decs[prec].init_weights(seed=1)
    cfg = S1.IMAGENET_S1
    P = {k: v.to(dev) for k, v in S1.make_params(cfg, seed=1).items()}
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = True, False
    arms = {"bf16": lambda: decs["bf16"].decode_code(ct, cb), "tf32": lambda: decs["tf32"].decode_code(ct, cb),
            "pytorch": lambda: S1.decode_code(P, cfg, ct, cb)}
    for f in arms.values():                                   # warm-up: modules, cuDNN algorithm choice
        for _ in range(2):
            f()
    torch.cuda.synchronize()
    flops = decs["bf16"].last_conv_flops
    assert flops == decs["tf32"].last_conv_flops
    times = {k: [] for k in arms}
    for r in range(a.rounds):
        for name, f in arms.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(a.iters):
                f()
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / a.iters
            times[name].append(ms / B)
            print(json.dumps({"round": r, "arm": name, "batch": B, "ms_per_image": round(ms / B, 4)}), flush=True)
    summary = {"batch": B, "rounds": a.rounds, "iters": a.iters, **info,
               "conv_gflop_per_image": round(flops / B * 1e-9, 2)}
    for name, ts in times.items():
        med = statistics.median(ts)
        tf = flops / B / (med * 1e-3) * 1e-12
        summary[name] = {"ms_per_image_median": round(med, 4), "ms_per_image_min": round(min(ts), 4),
                         "ms_per_image_max": round(max(ts), 4), "conv_tflops": round(tf, 1),
                         "frac_of_datasheet": round(tf / DATASHEET_TFLOPS[name], 3)}
    summary["tf32_over_bf16"] = round(summary["tf32"]["ms_per_image_median"] / summary["bf16"]["ms_per_image_median"], 3)
    summary["pytorch_over_tf32"] = round(summary["pytorch"]["ms_per_image_median"] / summary["tf32"]["ms_per_image_median"], 3)
    print(json.dumps(summary), flush=True)


if __name__ == "__main__":
    main()
