"""-m gpu: `bench.py --dump-outputs` writes the code grids of the last timed step: a bench run's dump (kernel table on, so
its replay runs after the timed steps) equals that step re-sampled here from the same arguments - same weights,
conditioning and Philox key."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.gpu


def test_bench_dump_is_the_last_timed_step(tmp_path):
    import bench
    import hqtransformer_b200 as H
    B, steps, warmup = 8, 2, 1
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--batch", str(B), "--steps", str(steps),
           "--warmup", str(warmup), "--no-cpu-baseline", "--no-ref-gpu", "--dump-outputs", str(tmp_path)]
    res = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-2000:]
    model = H.ImageGPT2.from_config(os.path.join(ROOT, "hqtransformer_b200", "configs", bench.CONFIGS["imagenet_l12"]),
                                    device=0, precision="bf16", max_batch=B).eval()
    s2 = model.stage2
    cond = torch.randint(0, s2.n_classes, (B,), generator=torch.Generator().manual_seed(1234)).cuda()
    ct, cb = H.sampling_ihqgpt(s2, B, cond, seed=warmup + steps - 1, use_fp16=True, max_seq_len=64, is_tqdm=False)
    assert sorted(os.listdir(tmp_path)) == ["codes_bot.npy", "codes_top.npy"]
    assert np.array_equal(np.load(tmp_path / "codes_top.npy"), ct.cpu().numpy().astype(np.float32))
    assert np.array_equal(np.load(tmp_path / "codes_bot.npy"), cb.cpu().numpy().astype(np.float32))
