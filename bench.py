#!/usr/bin/env python
"""bench.py - throughput of the HQ-Transformer hierarchical sampling loop (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # this repo's sm_100a engine
    python bench.py --impl reference --gpus N --steps K ...   # the reference algorithm on the host CPU cores

A "step" is one pass of the hot path over one batch: `sampling_ihqgpt` for `--batch` images per GPU, all 64 top
positions (320 codes per image), random-init weights of the named architecture (the reference's own
`measure_throughput` protocol: config only, no checkpoint; top-k/top-p None, T = 1, measure_throughput/__main__.py:93-104).
Weak scaling: the per-GPU batch is fixed, ranks share nothing but one final all-gather of the code grids.
Prints ONE JSON line on rank 0.  `--dump-outputs DIR` also writes the code grids of the last timed step (float32 .npy);
inputs, weights and Philox keys depend only on the arguments, so two builds run with the same arguments can be compared
output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "images_per_sec_sampled_256x256"
UNIT = "images/s"
CONFIGS = {"imagenet_l12": "imagenet_l12.yaml", "imagenet_l24": "imagenet_l24.yaml", "imagenet_l42": "imagenet_l42.yaml",
           "cc15m_l12": "cc15m_l12.yaml", "ffhq_l24": "ffhq_l24.yaml"}


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5, help="timed steps; --impl reference times at most 3 when it falls back to "
                    "the oracle port, and fewer when --ref-budget-s runs out (its JSON line reports both counts)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="graft", choices=["graft", "reference"])
    ap.add_argument("--model", default="imagenet_l12", choices=sorted(CONFIGS))
    ap.add_argument("--batch", type=int, default=256, help="images per GPU per step")
    ap.add_argument("--top-k", type=int, default=0, help="0 = None (measure_throughput protocol)")
    ap.add_argument("--top-p", type=float, default=0.0, help="0 = None")
    ap.add_argument("--temperature", type=float, default=1.0)
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-pdl", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-kernel-table", action="store_true")
    ap.add_argument("--cpu-batch", type=int, default=16, help="cpu_baseline leg of the default run: images per step")
    ap.add_argument("--cpu-positions", type=int, default=4, help="cpu_baseline leg of the default run: top positions per step")
    ap.add_argument("--ref-batch", type=int, default=64, help="--impl reference: images per step (all 64 positions)")
    ap.add_argument("--ref-budget-s", type=float, default=150.0, help="--impl reference: wall-clock budget of the timed steps")
    ap.add_argument("--no-ref-gpu", action="store_true", help="skip extras.reference_gpu_fp16_autocast")
    ap.add_argument("--ref-gpu-batch", type=int, default=0, help="batch of the reference-on-GPU extra (0 = --batch)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the code grids of the last timed step as DIR/<name>.npy (float32) for output comparison")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be >= 1")
    if args.dump_outputs and args.impl != "graft":
        ap.error("--dump-outputs applies to --impl graft")
    return args


DUMP_LIMIT_BYTES = (64 << 20) - 4096        # 64 MB in all, less room for the .npy headers


def dump_outputs(out_dir: str, arrays: dict) -> None:
    """Writes each [rows, ...] array as out_dir/<name>.npy in float32 (the codes are integers < 2^24, exact in it).
    When all of them together exceed DUMP_LIMIT_BYTES, the same fixed, seeded sample of rows is taken from each, and
    the sorted row indices go to out_dir/sampled_rows.npy."""
    import numpy as np
    import torch
    rows = next(iter(arrays.values())).shape[0]
    row_bytes = sum(t[0].numel() * 4 for t in arrays.values())
    keep = None
    if rows * row_bytes > DUMP_LIMIT_BYTES:
        n = DUMP_LIMIT_BYTES // (row_bytes + 4)     # + 4: the row's index in sampled_rows.npy
        keep = torch.randperm(rows, generator=torch.Generator().manual_seed(0))[:n].sort().values
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        t = t.detach().cpu()
        np.save(os.path.join(out_dir, f"{name}.npy"), (t if keep is None else t[keep]).numpy().astype(np.float32))
    if keep is not None:
        np.save(os.path.join(out_dir, "sampled_rows.npy"), keep.numpy().astype(np.float32))


# ---------------------------------------------------------------------------------------------------------------------
# clocks
# ---------------------------------------------------------------------------------------------------------------------
class ClockSampler:
    """Samples SM clocks and throttle reasons of one GPU while the timed region runs: NVML in-process every 20 ms (a short
    timed region still gets samples), `nvidia-smi -lms 100` as the fallback."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    NVML_REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None
        self.nvml, self.handle, self.stop_flag, self.sm, self.mx, self.reasons = None, None, False, [], None, set()

    def _nvml_loop(self):
        n = self.nvml
        while not self.stop_flag:
            try:
                self.sm.append(float(n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM)))
                bits = int(n.nvmlDeviceGetCurrentClocksEventReasons(self.handle)) if hasattr(n, "nvmlDeviceGetCurrentClocksEventReasons") \
                    else int(n.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle))
                for bit, name in self.NVML_REASONS.items():
                    if bits & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.02)

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            # NVML indexes physical devices: map the CUDA ordinal through CUDA_VISIBLE_DEVICES when it lists indices
            vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
            phys = self.index
            if vis and all(v.strip().isdigit() for v in vis.split(",")):
                phys = int(vis.split(",")[self.index])
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.mx = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
            self.nvml = pynvml
            self.thread = threading.Thread(target=self._nvml_loop, daemon=True)
            self.thread.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.nvml is not None:
            self.stop_flag = True
            self.thread.join(timeout=1)
            sm = sorted(self.sm)
            return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": self.mx, "samples": len(sm),
                    "reasons": sorted(self.reasons), "how": "NVML, 20 ms period"}
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = float(r[1])
            except Exception:
                continue
            for n, v in zip(names, r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "samples": len(sm), "reasons": sorted(reasons),
                "how": "nvidia-smi -lms 100"}


# ---------------------------------------------------------------------------------------------------------------------
# CPU arm: the reference algorithm (oracle port; /root/reference does not exist on the GPU box) on the host cores
# ---------------------------------------------------------------------------------------------------------------------
def cpu_reference_rate(model_name: str, batch: int, positions: int, steps: int, warmup: int):
    """images/s of the reference sampling algorithm on the host CPU: oracle/hq_oracle.py (fp32, torch CPU kernels with
    every host thread) run for `positions` of the 64 top positions on `batch` images; rate extrapolated linearly in
    positions (per-position cost is weight-bound and nearly flat in the cache length at these sizes)."""
    import torch
    from oracle import hq_oracle as O
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    cfg = {"imagenet_l12": O.IMAGENET_L12, "imagenet_l24": O.IMAGENET_L24, "imagenet_l42": O.IMAGENET_L42,
           "cc15m_l12": O.CC15M_L12}[model_name]
    P = O.make_params(cfg, seed=0, init="reference")
    g = torch.Generator().manual_seed(0)
    if cfg.cond == "txt":
        cond = torch.randint(0, cfg.vocab_txt, (batch, cfg.ctx_len_txt), generator=g)
    else:
        cond = torch.randint(0, cfg.n_classes, (batch,), generator=g)
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        O.sample(P, cfg, cond, batch, max_seq_len=positions, generator=g)
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
    sec = sum(times) / len(times)
    rate = batch * (positions / 64.0) / sec
    return rate, sec, cores, (f"{model_name} fp32, oracle port of the reference sampler, batch {batch}, {positions} of 64 top "
                              f"positions per step (rate scaled by {positions}/64), {len(times)} timed steps")


def _oracle_cfg(model_name: str):
    from dataclasses import replace
    from oracle import hq_oracle as O
    return {"imagenet_l12": O.IMAGENET_L12, "imagenet_l24": O.IMAGENET_L24, "imagenet_l42": O.IMAGENET_L42,
            "cc15m_l12": O.CC15M_L12,
            "ffhq_l24": replace(O.IMAGENET_L24, embed_dim=1024, n_heads=16, cond="uncond", embedding_type="reduce")}[model_name]


def reference_cpu_rates(model_name: str, plan, budget_s: float):
    """The UNMODIFIED reference sampler (`sampling_ihqgpt` -> `iHQGPT.sampling_step`, imported through oracle/ref_shim.py
    from the verbatim copy under baseline/_ref/) on the host CPU cores: fp32 (`use_fp16=False`, the reference's CPU mode),
    its own random init, measure_throughput protocol (one class per batch, top-k / top-p None, T = 1), ALL 64 top
    positions per step.  plan = [(batch, steps, warmup), ...]; returns {batch: (images/s, s/step, steps timed)} - at most
    `steps` steps per batch size, fewer when `budget_s` runs out (what was really timed is what is reported)."""
    import random
    import torch
    from oracle import ref_shim as R
    torch.set_num_threads(os.cpu_count() or 1)
    cfg = _oracle_cfg(model_name)
    model = R.build_reference_model_random(cfg)
    out = {}
    t_begin = time.perf_counter()
    for B, steps, warmup in plan:
        def one():
            if cfg.cond == "txt":
                cond = torch.randint(0, cfg.vocab_txt, (B, cfg.ctx_len_txt))
            else:
                cond = random.randint(0, cfg.n_classes - 1)
            t0 = time.perf_counter()
            ct, cb = R.reference_sample(model, B, cond, top_k_top=None, top_p_top=None, top_k_bot=None, top_p_bot=None,
                                        softmax_temperature=[1.0, 1.0], max_seq_len=64)
            assert tuple(ct.shape) == (B, 64) and tuple(cb.shape) == (B, 64, 4)
            return time.perf_counter() - t0
        for _ in range(warmup):
            one()
        times = []
        for _ in range(steps):
            times.append(one())
            if time.perf_counter() - t_begin > budget_s:
                break
        sec = sum(times) / len(times)
        out[B] = (B / sec, sec, len(times))
    return out


def run_reference_arm(args, rank: int):
    """`--impl reference`: the reference's own CPU implementation of the path on the box's host cores (rank 0 only)."""
    if rank != 0:
        return
    from oracle import ref_shim as R
    cores = os.cpu_count() or 1
    B = args.ref_batch
    if R.reference_available():
        kind = "reference"
        plan = [(B, args.steps, min(args.warmup, 1))] + [(b, 1, 0) for b in (4, 16) if b != B]   # BASELINE.md 3: B in {4, 16, 64}
        rates = reference_cpu_rates(args.model, plan, budget_s=args.ref_budget_s)
        rate, sec, timed = rates[B]
        extra = {f"B{b}": {"images_per_s": r[0], "s_per_step": r[1]} for b, r in rates.items() if b != B}
        sample = (f"{args.model}: UNMODIFIED reference sampler (sampling_ihqgpt, baseline/_ref copy) fp32 on {cores} host "
                  f"threads, batch {B}, all 64 top positions per step, own random init, {timed} timed step(s)")
        positions = 64
    else:       # no copy of the reference on this box: the oracle port on a bounded sample
        kind = "port"
        rate, sec, cores, sample = cpu_reference_rate(args.model, args.cpu_batch, args.cpu_positions, max(1, min(args.steps, 3)),
                                                      min(args.warmup, 1))
        timed, extra, positions, B = max(1, min(args.steps, 3)), {}, args.cpu_positions, args.cpu_batch
    line = {"impl": "reference", "metric": METRIC, "value": rate, "unit": UNIT, "n_gpus": args.gpus, "steps": timed,
            "steps_requested": args.steps, "warmup": min(args.warmup, 1), "ms_per_step": sec * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"{args.model}: {_oracle_cfg(args.model).cond}-conditional HQ-Transformer sampling, 64 top positions x (1 top + 4 "
                                   f"bottom codes), random-init weights, top_k=None top_p=None T=1.0; CPU sample: batch {B}, "
                                   f"{positions} positions per step",
                       "model": args.model, "batch": B, "positions": positions, "same_config_as_gpu_arm": False,
                       "note": "the GPU arm runs batch 256 per GPU; the reference on CPU is timed on a bounded batch"},
            "cpu_baseline": {"value": rate, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample, "other_batches": extra},
            "e2e": {"value": rate, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def reference_gpu_rate(model_name: str, B: int, device, steps: int = 2):
    """The honest "before" number: the UNMODIFIED reference sampler in its native mode on this same GPU - fp16 autocast,
    PyTorch eager, measure_throughput protocol (measure_throughput/__main__.py:93-104).  Returns a dict for `extras`."""
    import random
    import torch
    from oracle import ref_shim as R
    if not R.reference_available():
        return {"unavailable": "no copy of the reference under baseline/_ref on this box"}
    cfg = _oracle_cfg(model_name)
    try:
        model = R.build_reference_model_random(cfg).to(device)
        def one():
            cond = (torch.randint(0, cfg.vocab_txt, (B, cfg.ctx_len_txt)) if cfg.cond == "txt"
                    else random.randint(0, cfg.n_classes - 1))
            return R.reference_sample(model, B, cond, device="cuda", use_fp16=True, top_k_top=None, top_p_top=None,
                                      top_k_bot=None, top_p_bot=None, softmax_temperature=[1.0, 1.0], max_seq_len=64)
        with torch.no_grad():
            one()
            torch.cuda.synchronize(device)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                ct, _ = one()
            e1.record()
            torch.cuda.synchronize(device)
        ms = e0.elapsed_time(e1) / steps
        del model
        torch.cuda.empty_cache()
        return {"value": B / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms, "ms_per_top_position": ms / 64, "batch": B,
                "steps": steps, "what": "unmodified reference sampler (PyTorch eager, torch.cuda.amp.autocast fp16) on the "
                                        "same B200, same protocol and batch; baseline/_ref copy via oracle/ref_shim.py"}
    except Exception as e:      # a reference that cannot run on this torch / GPU must not take the bench line down
        return {"unavailable": f"{type(e).__name__}: {e}"[:300]}


def stage1_decode_extra(device, peaks, B: int = 32, iters: int = 5):
    """SURVEY.md 8f-1 beside the headline: stage-1 decode of code grids (the "decode" half of measure_throughput's total)
    through hq_s1_decode_codes - the shipped HQ-VAE decoder, random-init weights, batch `B` per call - and the UNMODIFIED
    reference `decode_code` (baseline/_ref copy, PyTorch eager / cuDNN) on the same GPU, one image at a time as
    measure_throughput/__main__.py:108-111 calls it, and batched."""
    import torch
    import hqtransformer_b200 as H
    out = {}
    try:
        dec = H.HQVAEDecoder(max_batch=B, device=device.index or 0)
        dec.init_weights(seed=1)
        ct = torch.randint(0, 8192, (B, 8, 8), device=device)
        cb = torch.randint(0, 8192, (B, 16, 16), device=device)
        for _ in range(2):
            dec.decode_code(ct, cb)
        torch.cuda.synchronize(device)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            dec.decode_code(ct, cb)
        e1.record()
        torch.cuda.synchronize(device)
        ms = e0.elapsed_time(e1) / iters
        tf = dec.last_conv_flops / (ms * 1e-3) * 1e-12
        out = {"value": B / (ms * 1e-3), "unit": "images/s decoded (256x256)", "ms_per_image": ms / B, "batch": B,
               "roofline": {"bound": "tensor", "kernel": "conv_tc2_kernel (all convolutions of a decode)", "achieved": tf,
                            "peak": peaks["bf16_tflops_sustained"], "unit": "TFLOP/s", "frac": tf / peaks["bf16_tflops_sustained"],
                            "note": "2 x MACs of the convolutions over interior pixels / WHOLE decode time (GroupNorm, attention, "
                                    "resampling included in the denominator)"},
               "what": "hq_s1_decode_codes: implicit-GEMM tcgen05 convolutions, bf16 inputs / fp32 accumulate and residual stream"}
        dec.close()
        del dec
        torch.cuda.empty_cache()
    except Exception as e:
        return {"unavailable": f"{type(e).__name__}: {e}"[:300]}
    try:
        from oracle import ref_shim as R, s1_oracle as S1
        if R.reference_available():
            model = R.build_reference_stage1(S1.IMAGENET_S1, S1.make_params(S1.IMAGENET_S1, seed=2)).to(device)
            ref = {}
            with torch.no_grad():
                for name, chunks, n in (("one_image_at_a_time", 8, 8), ("batched", 1, B)):
                    a, b = ct[:n].chunk(chunks), cb[:n].chunk(chunks)
                    run = lambda: [model.decode_code(x, y) for x, y in zip(a, b)]
                    run()
                    torch.cuda.synchronize(device)
                    e0.record()
                    for _ in range(2):
                        run()
                    e1.record()
                    torch.cuda.synchronize(device)
                    ref[name] = {"ms_per_image": e0.elapsed_time(e1) / 2 / n, "images_per_s": n / (e0.elapsed_time(e1) / 2 * 1e-3)}
            out["reference_same_gpu"] = dict(ref, what="unmodified SimRQGAN2Generator.decode_code, PyTorch eager (cuDNN, fp32 / TF32)")
            del model
            torch.cuda.empty_cache()
    except Exception as e:
        out["reference_same_gpu"] = {"unavailable": f"{type(e).__name__}: {e}"[:300]}
    return out


# ---------------------------------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------------------------------
def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"], "bf16_tflops_sustained": d["bf16_tflops_sustained"],
                "source": "measured (MEASURED_PEAKS.json)"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback (B200_PROFILING.md)"}


def kernel_table(eng, sp, B, cond_dev, ct, cb, D, peaks, p0=30, p1=34):
    """Per-kernel-family durations measured LIVE inside the real loop: hq_trace_run replays positions [p0, p1) of the
    batch just sampled with every kernel stamping %globaltimer (first CTA start -> last CTA end, device clock), i.e. the
    same launches, operands, cache state and CUDA-graph replay as the timed region.  Algorithmic work per launch:
    GEMM flops = 2 M N K, weight bytes = 2 N K; decode attention bytes = B * (2 * keys * D + 2 * D) * 2 (K and V rows of
    the cache once, q in, out)."""
    tl = eng.trace_run(batch=B, seq_len=64, pos_begin=p0, pos_end=p1, sampling=sp, cond=cond_dev, codes_top=ct, codes_bot=cb)
    npos = p1 - p0
    span_us = (max(e for _, _, e in tl) - min(s for _, s, _ in tl)) / 1e3 / npos
    fam = {}
    for tag, s, e in tl:
        f = fam.setdefault(tag, {"n": 0, "us": 0.0})
        f["n"] += 1
        f["us"] += (e - s) / 1e3
    rows = []
    for tag, f in fam.items():
        us = f["us"] / f["n"]
        row = {"kernel": tag, "launches_per_position": f["n"] / npos, "us": us, "us_per_position": f["us"] / npos,
               "share": f["us"] / npos / span_us}
        parts = tag.split(":")
        if parts[0].startswith("gemm") and len(parts) >= 2:
            M, N, K = (int(v) for v in parts[1].split("x"))
            splits = int(parts[2][1:]) if len(parts) > 2 else 1
            flops, wbytes = 2.0 * M * N * K, 2.0 * N * K
            row.update({"tflops": flops / us * 1e-6, "frac_tensor": flops / us * 1e-6 / peaks["bf16_tflops_sustained"],
                        "weight_gbs": wbytes / us * 1e-3, "frac_hbm": wbytes / us * 1e-3 / peaks["hbm_gbs"],
                        "splits": splits, "flops": flops, "bytes": wbytes})
        elif parts[0] == "attention_decode":
            keys = int(parts[1][1:])
            byt = B * (2.0 * keys * D + 2.0 * D) * 2.0
            row.update({"keys": keys, "gbs": byt / us * 1e-3, "frac_hbm": byt / us * 1e-3 / peaks["hbm_gbs"], "bytes": byt})
        rows.append(row)
    return rows, span_us


def run_graft_arm(args, rank: int, world: int, local_rank: int):
    import torch
    import torch.distributed as dist
    import hqtransformer_b200 as H
    from hqtransformer_b200.distributed import gather_codes
    from hqtransformer_b200.engine import SamplingParams

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    B = args.batch
    cfg_path = os.path.join(ROOT, "hqtransformer_b200", "configs", CONFIGS[args.model])
    model = H.ImageGPT2.from_config(cfg_path, device=local_rank, precision="bf16", max_batch=B,
                                    use_cuda_graph=not args.no_graph, use_pdl=not args.no_pdl).eval()
    s2 = model.stage2
    eng = s2.engine("bf16")
    g = torch.Generator().manual_seed(1234 + rank)
    if s2.use_txt_cond:
        cond_host = torch.randint(0, s2.vocab_size_txt, (B, s2.ctx_len_txt), generator=g)
    else:
        cond_host = torch.randint(0, s2.n_classes, (B,), generator=g)       # one class per row
    cond_dev = cond_host.to(dev)
    S = 64
    kw = dict(top_k_top=args.top_k or None, top_k_bot=args.top_k or None, top_p_top=args.top_p or None,
              top_p_bot=args.top_p or None, softmax_temperature=[args.temperature, args.temperature],
              use_fp16=True, max_seq_len=S, is_tqdm=False)

    local = {}

    def step(i):
        ct, cb = H.sampling_ihqgpt(s2, B, cond_dev, seed=i, row_offset=rank * B, **kw)
        local["ct"], local["cb"] = ct, cb
        if world > 1:
            ct, cb = gather_codes(ct, cb, world * B)     # the path's only collective: all-gather of the code grids
        return ct, cb

    def note(msg):
        if rank == 0:
            print(f"[bench] {msg}", file=sys.stderr, flush=True)

    note("model built; warming up")
    for i in range(args.warmup):
        step(i)
        torch.cuda.synchronize()
        note(f"warm-up step {i} done")
    if world > 1:
        dist.barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for i in range(args.steps):
        ct, cb = step(args.warmup + i)
    e1.record()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    ms = e0.elapsed_time(e1)
    clocks = sampler.stop()
    note(f"timed region done: {ms / args.steps:.1f} ms/step")
    launches = eng.last_launch_count * args.steps
    assert int(ct.min()) >= 0 and int(ct.max()) < s2.vocab_size_top and tuple(ct.shape) == (world * B, S)
    if args.dump_outputs and rank == 0:
        # now, before the kernel table's replay writes into these buffers again
        dump_outputs(args.dump_outputs, {"codes_top": ct, "codes_bot": cb})
        note(f"outputs of the last timed step written to {args.dump_outputs}")

    # ---- sharding invariance, checked on the grids of the last timed step: rank 0 re-samples ANOTHER shard of the global
    #      batch on its own GPU (that shard's conditioning, its global row offset, the same Philox key) and compares it
    #      bit for bit with the rows the all-gather delivered.  N = 1: rows [B/4, B/2) re-sampled as a shard of their own
    #      (another GEMM kernel: single CTA instead of CTA pairs). ----
    sharded_equal = None
    if rank == 0:
        last_seed = args.warmup + args.steps - 1
        if world > 1:
            other = 1
            g_o = torch.Generator().manual_seed(1234 + other)
            if s2.use_txt_cond:
                cond_o = torch.randint(0, s2.vocab_size_txt, (B, s2.ctx_len_txt), generator=g_o).to(dev)
            else:
                cond_o = torch.randint(0, s2.n_classes, (B,), generator=g_o).to(dev)
            ct_o, cb_o = H.sampling_ihqgpt(s2, B, cond_o, seed=last_seed, row_offset=other * B, **kw)
            sharded_equal = bool(torch.equal(ct_o, ct[other * B:(other + 1) * B]) and
                                 torch.equal(cb_o, cb[other * B:(other + 1) * B]))
        else:
            lo, hi = B // 4, B // 2
            if hi > lo:
                ct_o, cb_o = H.sampling_ihqgpt(s2, hi - lo, cond_dev[lo:hi], seed=last_seed, row_offset=lo, **kw)
                sharded_equal = bool(torch.equal(ct_o, ct[lo:hi]) and torch.equal(cb_o, cb[lo:hi]))
        note(f"sharded_equals_single: {sharded_equal}")

    # ---- end to end through the C-ABI host call: pinned host buffers, H2D of the conditioning and D2H of the grids
    #      inside the timed region ----
    cond_pin = cond_host.clone().pin_memory()
    ct_pin = torch.empty(B, S, dtype=torch.int64).pin_memory()
    cb_pin = torch.empty(B, S, 4, dtype=torch.int64).pin_memory()
    sp = SamplingParams(args.top_k or None, args.top_p or None, args.top_k or None, args.top_p or None,
                        args.temperature, args.temperature, seed=0, row_offset=rank * B)

    def e2e_step(i):
        sp.seed = i
        eng.run(batch=B, seq_len=S, pos_begin=0, pos_end=S, sampling=sp, cond=cond_pin, codes_top=ct_pin,
                codes_bot=cb_pin, host=True)

    e2e_step(0)
    torch.cuda.synchronize()
    note("e2e warm-up done")
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    for i in range(args.steps):
        e2e_step(1 + i)
    torch.cuda.synchronize()
    e2e_ms = (time.perf_counter() - t0) * 1e3
    if world > 1:
        t = torch.tensor([ms, e2e_ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, e2e_ms = float(t[0]), float(t[1])
    h2d = cond_pin.numel() * 8 + 48
    d2h = ct_pin.numel() * 8 + cb_pin.numel() * 8

    peaks = load_peaks()
    line = {"metric": METRIC, "value": world * B * args.steps / (ms * 1e-3), "unit": UNIT, "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": f"{args.model}: {s2.cond}-conditional HQ-Transformer sampling, 64 top positions x (1 top + 4 bottom "
                                   f"codes), batch {B} per GPU, random-init weights, top_k={args.top_k or None} "
                                   f"top_p={args.top_p or None} T={args.temperature}",
                       "model": args.model, "batch_per_gpu": B, "global_batch": world * B, "positions": S,
                       "parallelism": f"batch-sharded x{world}, one all-gather of code grids",
                       "cuda_graph": not args.no_graph, "pdl": not args.no_pdl,
                       "l2": "working set (weights + KV cache > 2 GB) exceeds the 126 MB L2; no explicit flush"},
            "ms_per_top_position": ms / args.steps / S,
            "e2e": {"value": world * B * args.steps / (e2e_ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h},
            "gpu_launches": launches, "clocks": clocks, "device_bytes": eng.device_bytes,
            "sharded_equals_single": sharded_equal,
            "parity_note": "bf16 tcgen05 engine: validated by teacher-forced logits against the reference / oracle within the "
                           "stated bf16 tolerance; bit-exact greedy grids vs the reference are shown for the fp32 engine "
                           "(tests/test_gpu_sampling_loop.py, tests/test_gpu_full_size.py)"}

    if rank == 0:
        D = s2.embed_dim
        local_ct, local_cb = local["ct"], local["cb"]
        if not args.no_kernel_table:
            rows, span_us = kernel_table(eng, sp, B, cond_dev, local_ct, local_cb, D, peaks)
            traffic = {}
            tp = os.path.join(ROOT, "profiles", "r2_ncu_traffic.json")
            if os.path.isfile(tp):
                traffic = json.load(open(tp))
            traffic.pop("_source", None)
            gemm_rows = [r for r in rows if r["kernel"].startswith("gemm")]
            gemm_us = sum(r["us_per_position"] for r in gemm_rows)
            gemm_flops = sum(r["flops"] * r["launches_per_position"] for r in gemm_rows)
            gemm_bytes = sum(r["bytes"] * r["launches_per_position"] for r in gemm_rows)
            # dominant kernel = the GEMM launch type with the largest share of a top position
            dom = max(gemm_rows, key=lambda r: r["us_per_position"])
            line["roofline"] = {
                "bound": "tensor", "kernel": dom["kernel"], "achieved": dom["tflops"], "peak": peaks["bf16_tflops_sustained"],
                "unit": "TFLOP/s", "frac": dom["frac_tensor"],
                "traffic": traffic.get(dom["kernel"], {}).get("dram_bytes"),
                "algorithmic_bytes_per_launch": dom["bytes"], "algorithmic_flops_per_launch": dom["flops"],
                "us_per_launch": dom["us"], "share_of_step": dom["share"],
                "hbm_view": {"achieved_gbs": dom["weight_gbs"], "peak_gbs": peaks["hbm_gbs"], "frac": dom["frac_hbm"]},
                "peak_source": peaks["source"] + ", sustained figure (kernel timed inside a long step)",
                "note": "an M = 256 launch is neither tensor- nor HBM-bound: about half of it is dependency hand-over, first tile "
                        "and tail, the main loop runs at ~320 ns per 128 columns of K (DESIGN.md 3.1 / 4, profiles/r2_gemm_phases.txt); "
                        "roofline_gemm_all aggregates every tcgen05 GEMM launch of a position",
                "how": "device %globaltimer per launch inside the replayed loop (hq_trace_run), top positions 30-33; "
                       "traffic IMPORTED from profiles/r2_ncu_traffic.json (ncu --set full capture of the same command, "
                       "committed; not measured in this run)"}
            line["roofline_gemm_all"] = {
                "bound": "tensor", "kernel": "all tcgen05 GEMM launches of a top position", "achieved": gemm_flops / gemm_us * 1e-6,
                "peak": peaks["bf16_tflops_sustained"], "unit": "TFLOP/s",
                "frac": gemm_flops / gemm_us * 1e-6 / peaks["bf16_tflops_sustained"], "share_of_step": gemm_us / span_us,
                "weight_stream_gbs": gemm_bytes / gemm_us * 1e-3}
            att = [r for r in rows if r["kernel"].startswith("attention_decode")]
            if att:
                att_us = sum(r["us_per_position"] for r in att)
                a_bytes = sum(r["bytes"] * r["launches_per_position"] for r in att)
                line["roofline_attention"] = {
                    "bound": "hbm", "kernel": "attention_decode_mma_kernel", "achieved": a_bytes / att_us * 1e-3,
                    "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": a_bytes / att_us * 1e-3 / peaks["hbm_gbs"],
                    "traffic": traffic.get("attention_decode:t64:B256", {}).get("dram_bytes"),
                    "traffic_note": "ncu capture at 64 keys (DRAM bytes vs 100.7 MB algorithmic); timed launches here have "
                                    + str(sorted(set(r["keys"] for r in att))) + " keys; a pure streaming kernel of the same "
                                    "access pattern and size (scripts/kv_stream_bench.cu, profiles/r1_kv_stream_bench.txt) needs "
                                    "about the same time: a cold 50 MB launch cannot reach the long-copy peak",
                    "share_of_step": att_us / span_us}
            line["kernels"] = [{k: (round(v, 4) if isinstance(v, float) else v) for k, v in r.items()
                                if k not in ("flops", "bytes")} for r in sorted(rows, key=lambda r: -r["us_per_position"])]
            line["trace_us_per_position"] = span_us
        if world == 1 and not args.no_cpu_baseline:
            rate, sec, cores, sample = cpu_reference_rate(args.model, args.cpu_batch, args.cpu_positions, 1, 1)
            line["cpu_baseline"] = {"value": rate, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample,
                                    "see_also": "`bench.py --impl reference` times the unmodified reference (kind \"reference\") "
                                                "over all 64 positions"}
        if world == 1 and not args.no_ref_gpu:
            del local_ct, local_cb
            line["extras"] = {"reference_gpu_fp16_autocast": reference_gpu_rate(args.model, args.ref_gpu_batch or B, dev),
                              "stage1_decode": stage1_decode_extra(dev, peaks)}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference_arm(args, rank)
        return
    if world != args.gpus and world == 1 and args.gpus > 1:
        # launched without torchrun: re-exec under torch.distributed.run so that `python bench.py --gpus N` works
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", os.environ.get("MASTER_PORT", "29511"), __file__] + sys.argv[1:]
        os.execv(sys.executable, cmd)
    run_graft_arm(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
