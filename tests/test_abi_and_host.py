"""not gpu: the C-ABI library loads and exports every declared symbol; host-side logic (config loading, sharding,
argument checks) behaves like the reference's; nothing here launches a kernel."""
import os
import re

import pytest
import torch

from oracle import ref_shim as R

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_symbol_the_header_declares():
    import ctypes
    from hqtransformer_b200 import _lib
    lib = _lib.load()
    header = open(os.path.join(ROOT, "include", "hqgraft.h")).read()
    declared = set(re.findall(r"^\s*(?:const\s+)?(?:int|int64_t|size_t|double|char\*|const char\*)\s+\*?(hq_[a-z_0-9]+)\s*\(", header, re.M))
    assert len(declared) >= 17, declared
    assert declared == set(_lib.PROTOTYPES), declared ^ set(_lib.PROTOTYPES)
    raw = ctypes.CDLL(_lib.LIB_PATH)
    for name in declared:
        assert hasattr(raw, name), f"{name} not exported"
    assert lib.hq_abi_version() == _lib.ABI_VERSION
    m = re.search(r"#define HQ_ABI_VERSION (\d+)", header)
    assert int(m.group(1)) == _lib.ABI_VERSION


def test_struct_layouts_match_header_sizes():
    import ctypes
    from hqtransformer_b200 import _lib
    assert ctypes.sizeof(_lib.HQConfig) == 22 * 4
    assert ctypes.sizeof(_lib.HQSamplingParams) == 56
    assert ctypes.sizeof(_lib.HQRunArgs) == 16 + 7 * 8 + 56 + 2 * 8 + 8


def test_philox_known_answers():
    """Random123 known-answer vectors for Philox4x32-10 (the engine's counter-based RNG; host build of the same code)."""
    from hqtransformer_b200.engine import debug_philox
    assert debug_philox(0, [0, 0, 0, 0]) == [0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8]
    assert debug_philox(0xffffffffffffffff, [0xffffffff] * 4) == [0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd]
    assert debug_philox(0x299f31d0a4093822, [0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344]) == \
        [0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1]


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU failure mode")
def test_no_cpu_fallback_create_fails_loudly_without_gpu():
    import hqtransformer_b200 as H
    with pytest.raises(H.HQError):
        H.Engine(embed_dim=128, n_heads=2, n_layers=1, n_layers_depth=1, vocab_top=64, vocab_bot=64, n_classes=10,
                 ctx_len_img=64, precision="fp32", max_batch=2)
    with pytest.raises(ValueError, match="CUDA"):
        H.Engine(embed_dim=128, n_heads=2, n_layers=1, n_layers_depth=1, vocab_top=64, vocab_bot=64, device="cpu")


def test_product_package_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "hqtransformer_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh")):
                src = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle", src, re.M), f
                assert "/root/reference" not in src, f


def test_config_loader_restates_reference_defaults():
    import hqtransformer_b200 as H
    from hqtransformer_b200.config import engine_kwargs
    cfg = H.load_config(os.path.join(ROOT, "hqtransformer_b200", "configs", "imagenet_l12.yaml"))
    s2 = cfg.stage2
    assert s2.ratio_bot2top == 4 and s2.vocab_size_txt == 16384 and s2.hparams_dec is None      # config2.py:85-105
    hp = s2.hparams
    assert (hp.embed_dim, hp.n_layers, hp.n_heads, hp.ctx_len_img, hp.n_classes) == (1536, 12, 24, 256, 1000)
    assert hp.position_embedding == "1d" and hp.mlp_bias and hp.attn_bias and hp.ctx_len_txt == 64   # config2.py:49-71
    kw = engine_kwargs(cfg)
    assert kw["model_type"] == "parallel" and kw["use_cls_cond"] and not kw["use_txt_cond"]
    l42 = H.load_config(os.path.join(ROOT, "hqtransformer_b200", "configs", "imagenet_l42.yaml"))
    assert l42.stage2.hparams.n_layers == 42 and l42.stage2.hparams_dec.n_layers == 6
    with pytest.raises(KeyError):
        H.merge_config({"stage2": {"type": "hq-transformer/parallel", "hparams": {"embed_dimm": 3}}})
    with pytest.raises(NotImplementedError):
        engine_kwargs(H.merge_config({"stage2": {"type": "top", "hparams": {}}}))


@pytest.mark.skipif(not os.path.isdir(os.path.join(R.REFERENCE_ROOT, "configs")),
                    reason="needs the original project's configs/ tree (HQ_REFERENCE_ROOT); not part of this repository")
def test_reference_yaml_files_load_unchanged():
    import hqtransformer_b200 as H
    from hqtransformer_b200.config import engine_kwargs
    base = os.path.join(R.REFERENCE_ROOT, "configs", "master", "stage2")
    for rel, L, Ld in (("imagenet/hqtransformer-embtrans1-soft1-layer12-top8x8.yaml", 12, None),
                       ("imagenet/hqtransformer-embtrans1-soft1-layer42-top8x8.yaml", 42, 6),
                       ("cc15m/hqtransformer-embtrans1-soft1-layer12-top8x8-cc15m.yaml", 12, None)):
        kw = engine_kwargs(H.load_config(os.path.join(base, rel)))
        assert kw["hparams"].n_layers == L and (kw["hparams_dec"].n_layers if kw["hparams_dec"] else None) == Ld


def test_shard_range_partitions_the_batch():
    from hqtransformer_b200.distributed import shard_range
    for B in (1, 7, 64, 256, 4096, 4097):
        for W in (1, 2, 4, 8):
            spans = [shard_range(B, r, W) for r in range(W)]
            assert spans[0][0] == 0 and spans[-1][1] == B
            assert all(spans[i][1] == spans[i + 1][0] for i in range(W - 1))
            sizes = [hi - lo for lo, hi in spans]
            assert max(sizes) - min(sizes) <= 1


def test_sampling_params_marshalling():
    from hqtransformer_b200.engine import SamplingParams
    c = SamplingParams(top_k_top=None, top_p_top=None, top_k_bot=2048, top_p_bot=1.0, temperature_top=0.95,
                       temperature_bot=0.9, seed=2 ** 64 + 5, row_offset=512).to_c()
    assert (c.top_k_top, c.top_k_bot) == (0, 2048) and c.top_p_top == 0.0 and c.top_p_bot == 1.0
    assert c.seed == 5 and c.row_offset == 512 and abs(c.temperature_top - 0.95) < 1e-7


def test_sampling_params_top_p_zero_is_keep_first():
    """The reference's nucleus cut with p = 0 keeps only the first sorted entry (utils/sampling.py:27-31); the ABI reserves
    0 for "no cut", so the host sends greedy."""
    from hqtransformer_b200.engine import SamplingParams
    c = SamplingParams(top_k_top=None, top_p_top=0.0, top_k_bot=50, top_p_bot=0.5).to_c()
    assert c.top_k_top == 1 and c.top_k_bot == 50 and abs(c.top_p_bot - 0.5) < 1e-7


def test_fresh_seed_follows_the_torch_generator():
    from hqtransformer_b200.models import fresh_seed
    torch.manual_seed(9)
    a, b = fresh_seed(), fresh_seed()
    torch.manual_seed(9)
    assert (a, b) == (fresh_seed(), fresh_seed()) and a != b and 0 <= a < 2 ** 63


def test_measure_throughput_cli_matches_the_reference_keys():
    """measure_throughput/__main__.py:34-48 fields as key=value; the README's `code-level` spelling is accepted too."""
    from hqtransformer_b200.measure_throughput import Experiment, parse_cli
    a = parse_cli(["model_path=x.yaml", "batch_size=32", "code-level=2"])
    assert (a.model_path, a.batch_size, a.code_levels, a.n_loop, a.warmup, a.top_resolution) == ("x.yaml", 32, 2, 6, 1, 8)
    assert Experiment().batch_size == 50
    with pytest.raises(SystemExit):
        parse_cli(["batch_size=3"])                    # model_path is required
    with pytest.raises(SystemExit):
        parse_cli(["model_path=x.yaml", "bogus=1"])


def test_graft_entry_build_is_idempotent():
    import __graft_entry__ as G
    G.build()
    assert os.path.isfile(os.path.join(ROOT, "hqtransformer_b200", "libhqgraft.so"))


def test_committed_bench_evidence_carries_the_contract_keys():
    """profiles/r1_bench_B256.json is the bench line the docs quote: it must hold every key of the bench contract
    (roofline with achieved / peak / frac / traffic for the dominant kernel, cpu_baseline, e2e with copy sizes, clocks,
    launch count), with internally consistent numbers."""
    import json
    import os
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    d = json.load(open(os.path.join(root, "profiles", "r1_bench_B256.json")))
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "dtype",
              "data", "config", "e2e", "gpu_launches", "clocks", "roofline", "cpu_baseline"):
        assert k in d, k
    assert d["metric"] == "images_per_sec_sampled_256x256" and d["unit"] == "images/s" and d["n_gpus"] == 1
    assert d["warmup"] >= 3 and d["config"]["batch_per_gpu"] == 256 and "workload" in d["config"]
    assert abs(d["value"] - 256 * d["steps"] / (d["ms_per_step"] * d["steps"] * 1e-3)) < 1e-6 * d["value"]
    r = d["roofline"]
    assert r["bound"] in ("hbm", "tensor") and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9 and r["traffic"] > 0
    assert d["e2e"]["h2d_bytes_per_step"] > 0 and d["e2e"]["d2h_bytes_per_step"] == 256 * 64 * 5 * 8
    assert d["gpu_launches"] == d["steps"] * 64 * 145
    assert d["cpu_baseline"]["kind"] in ("port", "reference") and d["cpu_baseline"]["cores"] >= 1
    assert not set(d["clocks"]["reasons"]) & {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"}
    ra = d["roofline_attention"]
    assert ra["bound"] == "hbm" and abs(ra["frac"] - ra["achieved"] / ra["peak"]) < 1e-9


def test_bench_dump_outputs_is_exact_and_samples_rows_over_the_limit(tmp_path, monkeypatch):
    """bench.py --dump-outputs: code grids round-trip exactly through float32 .npy; above the size limit every array keeps
    the same seeded sample of rows, listed in sampled_rows.npy."""
    import numpy as np
    import bench
    g = torch.Generator().manual_seed(0)
    ct, cb = torch.randint(0, 16384, (40, 64), generator=g), torch.randint(0, 16384, (40, 64, 4), generator=g)
    bench.dump_outputs(str(tmp_path / "all"), {"codes_top": ct, "codes_bot": cb})
    assert sorted(os.listdir(tmp_path / "all")) == ["codes_bot.npy", "codes_top.npy"]
    top = np.load(tmp_path / "all" / "codes_top.npy")
    assert top.dtype == np.float32 and np.array_equal(top, ct.numpy())
    assert np.array_equal(np.load(tmp_path / "all" / "codes_bot.npy"), cb.numpy())
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 10 * (64 + 256) * 4 + 40)
    for d in ("s1", "s2"):
        bench.dump_outputs(str(tmp_path / d), {"codes_top": ct, "codes_bot": cb})
    rows = np.load(tmp_path / "s1" / "sampled_rows.npy").astype(np.int64)
    assert len(rows) == 10 and np.all(np.diff(rows) > 0)
    assert np.array_equal(rows, np.load(tmp_path / "s2" / "sampled_rows.npy").astype(np.int64))
    assert np.array_equal(np.load(tmp_path / "s1" / "codes_top.npy"), ct.numpy()[rows])
    assert np.array_equal(np.load(tmp_path / "s1" / "codes_bot.npy"), cb.numpy()[rows])


def test_encode_prompts_pads_and_truncates_like_the_reference_dataset():
    """hqvae/datasets/__init__.py:145-152: "[PAD]" padding to the context length + truncation, int64 [N, 64]."""
    tokenizers = pytest.importorskip("tokenizers")
    from tokenizers import Tokenizer, models, pre_tokenizers
    from hqtransformer_b200.sampling import encode_prompts
    vocab = {"[UNK]": 0, "a": 1, "photo": 2, "of": 3, "cat": 4, "dog": 5}
    tok = Tokenizer(models.WordLevel(vocab, unk_token="[UNK]"))
    tok.pre_tokenizer = pre_tokenizers.Whitespace()
    ids = encode_prompts(tok, ["a photo of a cat", "dog " * 100], context_length=8)
    assert ids.dtype == torch.int64 and tuple(ids.shape) == (2, 8)
    pad = tok.token_to_id("[PAD]")
    assert ids[0].tolist() == [1, 2, 3, 1, 4, pad, pad, pad] and ids[1].tolist() == [5] * 8
