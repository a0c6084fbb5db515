"""Drop-in for the reference's timing harness:

    python -m hqtransformer_b200.measure_throughput model_path=<stage2 yaml> [batch_size=50] [code_levels=2]

Same `key=value` command line, defaults, protocol and report as `measure_throughput/__main__.py` of the reference
(:34-48 the `Experiment` fields, :76 ceil(1000 / batch_size) iterations per loop, :93-104 the sampling call - random
class per iteration, top-k / top-p None, T = 1, fp16, 64 top positions -, :147-155 and :161-179 the report: n_loop loops
with the first `warmup` discarded, "ms/sample (ar: ..., decode: ...)").  `load_model` builds the model from the config
only, i.e. with random-init weights (:25-31).

The "ar" figure is the sampling loop, "decode" is stage 1 (`model.stage1.decode_code`, :106-113); both run in libhqgraft.
The reference decodes one image at a time (`codes.chunk(batch_size)`, :108-111); here the batch is decoded in one call
(`decode_chunks=1`; `decode_chunks=<batch_size>` reproduces the one-by-one protocol).  `stage1=0` skips the decoder.
The README of the reference spells the level key `code-level` (configs/README.md:70) while the dataclass field is
`code_levels` (:48); both are accepted.  code_levels=3 takes a `multilevel-hq` config (the 3-level `HQTransformer`,
configs/README.md:68-71) and times its sampler; the 3-level stage-1 decoder is not implemented, so "decode" is 0 there.
"""
from __future__ import annotations

import platform
import random
import sys
import time
from dataclasses import dataclass, fields

import torch

from .models import ImageGPT2
from .sampling import codes_to_grids, sampling_ihqgpt


@dataclass
class Experiment:                      # measure_throughput/__main__.py:34-48
    f: int = 32
    model: str = "huge"
    d: int = 4
    c: int = 16384
    batch_size: int = 50
    n_loop: int = 6
    warmup: int = 1
    model_path: str = ""
    top_resolution: int = 8
    code_levels: int = 2
    n_samples: int = 1000              # extension: images per loop (the reference hard-codes 1000, :76)
    stage1: int = 1                    # extension: 1 = build and time the stage-1 decoder too
    decode_chunks: int = 1             # extension: chunks the batch is decoded in (batch_size = the reference's protocol)
    precision: str = "bf16"            # extension: engine of use_fp16=True - "bf16", or "fp16" (the reference's autocast type)
    stage1_precision: str = "bf16"     # extension: stage-1 decoder format - "bf16", or "tf32" (the reference's decode format)


def parse_cli(argv) -> Experiment:
    """`OmegaConf.from_cli()` merged over the structured defaults (:185): `key=value` tokens, typed by the field."""
    args = Experiment()
    known = {f.name: f.type for f in fields(Experiment)}
    alias = {"code-level": "code_levels", "code_level": "code_levels", "code-levels": "code_levels"}
    for tok in argv:
        if "=" not in tok:
            raise SystemExit(f"expected key=value, got {tok!r}")
        k, v = tok.split("=", 1)
        k = alias.get(k, k)
        if k not in known:
            raise SystemExit(f"unknown key {k!r}; known: {sorted(known)}")
        setattr(args, k, type(getattr(args, k))(v))
    if not args.model_path:
        raise SystemExit("model_path=<stage2 yaml> is required")
    return args


def load_model(result_path: str, device="cuda", max_batch: int = 50, with_stage1: bool = True,
               precision: str = "bf16", stage1_precision: str = "bf16", max_seq_len: int = 64) -> ImageGPT2:
    """:25-31 - config only, no checkpoint: random-init weights of the named architecture.  max_seq_len: top positions the
    engine is built for (top_resolution ** 2 in the reference protocol)."""
    dev = torch.device(device)
    return ImageGPT2.from_config(result_path, device=dev.index or 0, precision=precision, max_batch=max_batch,
                                 with_stage1=with_stage1, stage1_max_batch=min(max_batch, 32), stage1_precision=stage1_precision,
                                 max_seq_len=max_seq_len)


def main(args: Experiment):
    torch.set_grad_enabled(False)
    if args.code_levels not in (2, 3):
        raise NotImplementedError("code_levels must be 2 (iHQGPT) or 3 (HQTransformer)")
    device = torch.device("cuda")
    if args.precision not in ("bf16", "fp16"):
        raise SystemExit(f"precision={args.precision!r}: bf16 or fp16 (the engines use_fp16=True selects)")
    if args.stage1_precision not in ("bf16", "tf32"):
        raise SystemExit(f"stage1_precision={args.stage1_precision!r}: bf16 or tf32")
    model_ar = load_model(args.model_path, device, args.batch_size,
                          with_stage1=bool(args.stage1) and args.code_levels == 2, precision=args.precision,
                          stage1_precision=args.stage1_precision,
                          max_seq_len=args.top_resolution * args.top_resolution).to(device).eval()
    if (args.code_levels == 3) != hasattr(model_ar.stage2, "code_level"):
        raise SystemExit(f"code_levels={args.code_levels} does not match the model type of {args.model_path}")
    title = f"bs{args.batch_size}, sampling loops {args.warmup + 1}-{args.n_loop}"
    print(title)
    print("python: %s, torch: %s, cudnn: %s, cuda: %s, gpu: %s" % (
        platform.python_version(), torch.__version__, torch.backends.cudnn.version(), torch.version.cuda,
        torch.cuda.get_device_name(device)))
    ar_size = sum(int(torch.tensor(s).prod()) for s in model_ar.stage2.param_shapes().values()) / 10 ** 6
    print(f"transformer size: {ar_size:.1f}M")
    batch_size = args.batch_size
    n_iter_per_loop = (args.n_samples + batch_size - 1) // batch_size
    n_loop = args.n_loop
    n_classes = model_ar.stage2.n_classes or 1000
    is_txt = model_ar.stage2.use_txt_cond
    from .hqtransformer3 import sampling_hqtransformer

    def loop(loop_idx: int):
        starts = [torch.cuda.Event(enable_timing=True) for _ in range(n_iter_per_loop)]
        middles = [torch.cuda.Event(enable_timing=True) for _ in range(n_iter_per_loop)]
        ends = [torch.cuda.Event(enable_timing=True) for _ in range(n_iter_per_loop)]
        torch.cuda.synchronize(device)
        tic = time.time()
        for i in range(n_iter_per_loop):
            starts[i].record()
            if is_txt:      # measure_throughput_txt/__main__.py:128-139: a [B, 64] batch of token ids
                cond = torch.randint(0, model_ar.stage2.vocab_size_txt, (batch_size, model_ar.stage2.ctx_len_txt), device=device)
            else:
                cond = random.randint(0, n_classes - 1)
            if args.code_levels == 3:     # measure_throughput/__main__.py:113-127: sampling_hqtransformer, top_k / top_p None
                sampling_hqtransformer(model_ar.stage2, num_candidates=batch_size, cond=cond, top_k=[None] * 3, top_p=[None] * 3,
                                       softmax_temperature=[1.0] * 3, use_fp16=True, is_tqdm=False,
                                       max_seq_len=args.top_resolution * args.top_resolution)
                middles[i].record()
                ends[i].record()
                continue
            codes_t, codes_b = sampling_ihqgpt(model_ar.stage2, cond=cond, num_candidates=batch_size, top_k_top=None,
                                               top_p_top=None, top_k_bot=None, top_p_bot=None,
                                               softmax_temperature=[1.0 for _ in range(args.code_levels)], use_fp16=True,
                                               is_tqdm=False, max_seq_len=args.top_resolution * args.top_resolution,
                                               model_stage1=None)
            middles[i].record()
            codes_t, codes_b = codes_to_grids(codes_t, codes_b, H=args.top_resolution)
            if model_ar.stage1 is not None:
                pixels = torch.cat([model_ar.stage1.decode_code(ct, cb)
                                    for ct, cb in zip(codes_t.chunk(args.decode_chunks), codes_b.chunk(args.decode_chunks))], dim=0)
                _ = (0.5 * pixels + 0.5).clamp(0, 1)
            ends[i].record()
        torch.cuda.synchronize(device)
        toc = time.time()
        elapsed_time = toc - tic
        elapsed_time_ar = sum(starts[i].elapsed_time(middles[i]) for i in range(n_iter_per_loop)) / 1000
        elapsed_time_decode = sum(middles[i].elapsed_time(ends[i]) for i in range(n_iter_per_loop)) / 1000
        print(f"{loop_idx + 1}/{n_loop} | {elapsed_time:.1f} s/loop (ar: {elapsed_time_ar:.1f}, decode: {elapsed_time_decode:.1f})")
        n = n_iter_per_loop * batch_size
        speed, speed_ar, speed_decode = (elapsed_time / n * 1000, elapsed_time_ar / n * 1000, elapsed_time_decode / n * 1000)
        print(f"{loop_idx + 1}/{n_loop} | {speed:.2f} ms/sample (ar: {speed_ar:.2f}, decode: {speed_decode:.2f})")
        return speed, speed_ar, speed_decode

    speeds, speeds_ar, speeds_decode = [], [], []
    print("-" * 80)
    for loop_idx in range(args.n_loop):
        speed, speed_ar, speed_decode = loop(loop_idx)
        if loop_idx < args.warmup:
            continue
        speeds.append(speed)
        speeds_ar.append(speed_ar)
        speeds_decode.append(speed_decode)
    print("-" * 80)
    n = len(speeds)
    speed, speed_ar, speed_decode = sum(speeds) / n, sum(speeds_ar) / n, sum(speeds_decode) / n
    print(f"{title} | {speed:.4f} ms/sample (ar: {speed_ar:.4f}, decode: {speed_decode:.4f})")
    print("=" * 80)
    return speed, speed_ar, speed_decode


if __name__ == "__main__":
    main(parse_cli(sys.argv[1:]))
