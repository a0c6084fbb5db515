"""Full-context sampling and larger stage-1 grids on the CPU: 16 x 16 grid layouts, the top_resolution field of
measure_throughput, the stage-1 oracle on larger grids and the new C ABI entry points."""
import ctypes
import os
import re

import pytest
import torch

from hqtransformer_b200 import _lib
from hqtransformer_b200.measure_throughput import parse_cli
from hqtransformer_b200.sampling import codes_to_grids, grids_to_codes
from oracle import s1_oracle as S1

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NEW_SYMBOLS = ("hq_s1_reserve_grid", "hq_s1_decode_codes_grid")


def test_grids_round_trip_at_16x16():
    g = torch.Generator().manual_seed(16)
    ct = torch.randint(0, 1 << 14, (3, 256), generator=g)
    cb = torch.randint(0, 1 << 14, (3, 256, 4), generator=g)
    t, b = codes_to_grids(ct, cb, H=16)
    assert tuple(t.shape) == (3, 16, 16) and tuple(b.shape) == (3, 32, 32)
    # raster position p is row p // 16, column p % 16
    assert int(t[1, 5, 9]) == int(ct[1, 5 * 16 + 9])
    ct2, cb2 = grids_to_codes(t, b)
    assert torch.equal(ct2, ct) and torch.equal(cb2, cb)


def test_measure_throughput_parses_top_resolution():
    args = parse_cli(["model_path=hqtransformer_b200/configs/imagenet_l12.yaml", "top_resolution=16"])
    assert args.top_resolution == 16 and isinstance(args.top_resolution, int)
    assert parse_cli(["model_path=x.yaml"]).top_resolution == 8


def test_s1_oracle_on_twice_the_grid():
    cfg = S1.TINY_S1
    P = S1.make_params(cfg, seed=0)
    h = cfg.latent_res                     # twice the configured top grid
    ct = torch.randint(0, cfg.n_embed, (1, h, h))
    cb = torch.randint(0, cfg.n_embed, (1, 2 * h, 2 * h))
    px = S1.decode_code(P, cfg, ct, cb)
    assert tuple(px.shape) == (1, cfg.out_ch, 2 * cfg.resolution, 2 * cfg.resolution)


def test_new_entry_points_in_header_binding_and_library():
    header = open(os.path.join(ROOT, "include", "hqgraft.h")).read()
    for name in NEW_SYMBOLS:
        assert re.search(r"\b%s\(" % name, header), name
        assert name in _lib.PROTOTYPES, name
    lib_path = os.path.join(ROOT, "hqtransformer_b200", "libhqgraft.so")
    lib = ctypes.CDLL(lib_path)
    for name in NEW_SYMBOLS:
        assert hasattr(lib, name), name
    assert lib.hq_abi_version() == 9
    # both reject a null context before touching a device
    lib.hq_s1_reserve_grid.argtypes = [ctypes.c_void_p, ctypes.c_int]
    assert lib.hq_s1_reserve_grid(None, 16) != 0
