"""not gpu: pins the oracle (oracle/hq_oracle.py) against the known answers produced by the UNMODIFIED reference
(tests/golden/*.npz, made by oracle/make_golden.py) and, when the reference's source tree is present, against the live
reference itself."""
import numpy as np
import pytest
import torch

from oracle import hq_oracle as O
from oracle import make_golden as G
from oracle import ref_shim as R
from tests.helpers import cfg_from_meta, load_golden

GREEDY = dict(top_k_top=1, top_p_top=1.0, top_k_bot=1, top_p_bot=1.0)


@pytest.mark.parametrize("name", ["tiny_cls_greedy.npz", "small_cls_greedy.npz", "asym_cls_greedy.npz"])
def test_oracle_greedy_codes_and_logits_equal_reference(name):
    g, meta = load_golden(name)
    assert meta["torch"].split("+")[0] == torch.__version__.split("+")[0], "goldens depend on torch's RNG stream"
    cfg = cfg_from_meta(meta)
    P = O.make_params(cfg, seed=meta["seed"], init=meta["init"])
    labels = torch.from_numpy(g["labels"])
    ct, cb, lg = O.sample(P, cfg, labels, len(labels), return_logits=True, **GREEDY)
    assert np.array_equal(ct.numpy(), g["codes_top"]) and np.array_equal(cb.numpy(), g["codes_bot"])
    got = lg[:, meta["logit_positions"]].numpy()
    assert np.abs(got - g["logits"]).max() < 1e-5
    assert meta["min_logit_margin"] >= 1e-4          # what makes the bit-exact GPU test meaningful
    # scalar class broadcast = the reference's own driver
    ct_s, cb_s = O.sample(P, cfg, int(labels[-1]), len(labels), **GREEDY)
    assert np.array_equal(ct_s.numpy(), g["codes_top_scalar_class"])
    assert np.array_equal(cb_s.numpy(), g["codes_bot_scalar_class"])


def test_oracle_equals_reference_at_imagenet_l12_size():
    """BASELINE config 1 at the reference's real scale: ImageNet-L12 architecture (530 M parameters), batch 4, greedy,
    64 positions - the grids the unmodified reference produced (tests/golden/l12_cls_greedy_b4.npz)."""
    g, meta = load_golden("l12_cls_greedy_b4.npz")
    cfg = cfg_from_meta(meta)
    assert cfg == O.IMAGENET_L12 and meta["min_logit_margin"] >= 1e-4
    P = O.make_params(cfg, seed=meta["seed"], init=meta["init"])
    labels = torch.from_numpy(g["labels"])
    ct, cb, lg = O.sample(P, cfg, labels, len(labels), return_logits=True, **GREEDY)
    assert np.array_equal(ct.numpy(), g["codes_top"]) and np.array_equal(cb.numpy(), g["codes_bot"])
    assert np.abs(lg[:, meta["logit_positions"]].numpy() - g["logits"]).max() < 1e-5


@pytest.mark.parametrize("name", ["tiny_txt_greedy.npz", "asym_txt_greedy.npz"])
def test_oracle_text_prefix_equals_reference(name):
    g, meta = load_golden(name)
    cfg = cfg_from_meta(meta)
    P = O.make_params(cfg, seed=meta["seed"], init=meta["init"])
    ids = torch.from_numpy(g["text_ids"])
    ct, cb = O.sample(P, cfg, ids, ids.shape[0], **GREEDY)
    assert np.array_equal(ct.numpy(), g["codes_top"]) and np.array_equal(cb.numpy(), g["codes_bot"])


def test_oracle_stochastic_sequence_equals_reference_under_shared_torch_seed():
    """Same torch generator state + same draw order (top, b0..b3 per position) -> identical sequences."""
    g, meta = load_golden("tiny_uncond_stochastic.npz")
    cfg = cfg_from_meta(meta)
    P = O.make_params(cfg, seed=meta["seed"], init=meta["init"])
    torch.manual_seed(meta["torch_seed"])
    ct, cb = O.sample(P, cfg, None, g["codes_top"].shape[0], top_k_top=meta["top_k_top"], top_p_top=meta["top_p_top"],
                      top_k_bot=meta["top_k_bot"], top_p_bot=meta["top_p_bot"],
                      softmax_temperature=meta["softmax_temperature"])
    assert np.array_equal(ct.numpy(), g["codes_top"]) and np.array_equal(cb.numpy(), g["codes_bot"])


def test_oracle_filters_equal_reference_known_answers():
    g, _ = load_golden("filters.npz")
    x = torch.from_numpy(g["topk_in"])
    for k in (1, 2, 5, 64, 512):
        assert np.array_equal(O.cutoff_topk_logits(x.clone(), k).numpy(), g[f"topk_{k}"])
    for key, pin in (("topp", "topp_in"), ("topp_small", "topp_small_in")):
        p_in = torch.from_numpy(g[pin])
        for p in (0.5, 0.8, 0.95, 1.0):
            np.testing.assert_allclose(O.cutoff_topp_probs(p_in.clone(), p).numpy(), g[f"{key}_{p}"], rtol=0, atol=1e-7)
    # the survey's worked example (SURVEY.md 8a a9)
    small = torch.tensor([[0.5, 0.3, 0.15, 0.05]])
    assert (O.cutoff_topp_probs(small, 0.8) > 0).sum() == 2 and (O.cutoff_topp_probs(small, 0.95) > 0).sum() == 3


def test_bf16_emulation_is_close_to_fp32_but_not_equal():
    g, meta = load_golden("tiny_cls_greedy.npz")
    cfg = cfg_from_meta(meta)
    P = O.make_params(cfg, seed=meta["seed"], init=meta["init"])
    labels = torch.from_numpy(g["labels"])[:2]
    ct, cb = torch.from_numpy(g["codes_top"])[:2, :4], torch.from_numpy(g["codes_bot"])[:2, :4]
    a = O.step_logits(P, cfg, labels, ct, cb)
    b = O.step_logits(P, cfg, labels, ct, cb, emulate="bf16")
    d = (a - b).abs().max().item()
    assert 0 < d < 0.15


def test_code_grid_layout():
    """'B (H W) (kerH kerW) -> B (H kerH) (W kerW)' (sampling_hqmodel.py:119-120) without einops."""
    ct = torch.arange(2 * 64).view(2, 64)
    cb = torch.arange(2 * 64 * 4).view(2, 64, 4)
    top, bot = O.codes_to_grids(ct, cb)
    assert tuple(top.shape) == (2, 8, 8) and tuple(bot.shape) == (2, 16, 16)
    from einops import rearrange
    assert torch.equal(top, rearrange(ct, "B (H W) -> B H W", H=8))
    assert torch.equal(bot, rearrange(cb, "B (H W) (kerH kerW) -> B (H kerH) (W kerW)", H=8, kerH=2))
    # position cnt, slot j lands at row 2*(cnt//8) + j//2, col 2*(cnt%8) + j%2
    assert bot[1, 2 * 3 + 1, 2 * 5 + 0] == cb[1, 3 * 8 + 5, 2]


def _check_seeded_runs(name, only=None):
    """The oracle against the stored grids of the seeded runs in tests/golden/<name> (oracle/make_golden.py LIVE_CHECKS),
    and against the live reference on the same runs when the tree is present."""
    g, meta = load_golden(name)
    assert meta["torch"].split("+")[0] == torch.__version__.split("+")[0], "seeded goldens depend on torch's RNG stream"
    runs = [r for r in meta["runs"] if only is None or only(r)]
    assert runs
    for run in runs:
        got = G.live_check_run(name, run)
        for level, codes in zip(("top", "mid", "bot") if len(got) == 3 else ("top", "bot"), got):
            assert np.array_equal(codes.numpy(), g[f"{run['run']}_{level}"]), (run["run"], level)
        if R.reference_available():
            assert all(torch.equal(a, b) for a, b in zip(got, G.live_check_run(name, run, reference=True))), run["run"]


def test_oracle_equals_live_reference_tiny():
    """The reference's own driver (sampling_ihqgpt + iHQGPT.sampling_step, one class for the whole batch): greedy, and
    stochastic with top-k / top-p and two temperatures under a fixed torch seed (tests/golden/tiny_cls_scalar_class.npz)."""
    _check_seeded_runs("tiny_cls_scalar_class.npz")


def test_teacher_forced_forward_matches_incremental_sampling():
    """Teacher forcing against incremental sampling (SURVEY.md 3.5): with the reference-made greedy grids forced as input,
    the argmax of every top and bottom logit is the forced code - through the oracle's teacher-forced pass, and, when the
    tree is present, through the reference's training-time forward() (a path the reference never runs while sampling)."""
    g, meta = load_golden("tiny_cls_greedy.npz")
    cfg = cfg_from_meta(meta)
    P = O.make_params(cfg, seed=meta["seed"], init=meta["init"])
    ct, cb = torch.from_numpy(g["codes_top"]), torch.from_numpy(g["codes_bot"])
    lg = O.step_logits(P, cfg, torch.from_numpy(g["labels"]), ct, cb)
    assert torch.equal(lg[:, :, 0, : cfg.vocab_top].argmax(-1), ct)
    assert torch.equal(lg[:, :, 1:, : cfg.vocab_bot].argmax(-1), cb)
    if not R.reference_available():
        return
    model = R.build_reference_model(cfg, P)
    _, bot_grid = O.codes_to_grids(ct, cb)
    with torch.no_grad():
        out = model((ct, bot_grid.reshape(ct.shape[0], -1)), torch.from_numpy(g["labels"]))
    logits_top, logits_bot = out[0], out[1]
    assert torch.equal(logits_top.argmax(-1), ct)


VARIANT_GOLDENS = ["tiny_reduce_uncond_greedy.npz", "tiny_pos2d_cls_greedy.npz", "tiny_top2bot_cls_greedy.npz",
                   "tiny_bidir_cls_greedy.npz", "asym_top2bot_reduce_pos2d_greedy.npz"]


@pytest.mark.parametrize("name", VARIANT_GOLDENS)
def test_oracle_model_variants_equal_reference(name):
    """SURVEY.md 8f-3: embedding_type 'reduce', position_embedding '2d', model_type 'top2bot' / 'bidirectional',
    unconditional sos - greedy grids of the unmodified reference (oracle/make_golden.py --variants)."""
    g, meta = load_golden(name)
    cfg = cfg_from_meta(meta)
    assert meta["min_logit_margin"] >= 1e-4
    P = O.make_params(cfg, seed=meta["seed"], init=meta["init"])
    B = g["codes_top"].shape[0]
    cond = torch.from_numpy(g["labels"]) if cfg.cond == "cls" else None
    ct, cb = O.sample(P, cfg, cond, B, **GREEDY)
    assert np.array_equal(ct.numpy(), g["codes_top"]) and np.array_equal(cb.numpy(), g["codes_bot"])


@pytest.mark.parametrize("kw", [dict(model_type="top2bot"), dict(model_type="bidirectional"),
                                dict(embedding_type="reduce", position_embedding="2d", cond="uncond")])
def test_oracle_variants_stochastic_equal_live_reference(kw):
    """Same torch seed, same draw order -> identical stochastic sequences ('bidirectional' draws every token with the
    bottom filters and softmax_temperature[0], hierarchical_ar.py:860-866); tests/golden/tiny_variants_stochastic.npz."""
    _check_seeded_runs("tiny_variants_stochastic.npz", only=lambda run: run["cfg"] == kw)


def test_stage1_oracle_equals_reference_golden_and_live_reference():
    """SURVEY.md 8f-1: oracle/s1_oracle.py against the pixels the unmodified SimRQGAN2Generator.decode_code produced for
    these same code grids and weights (tests/golden/s1_tiny_decode.npz), and against the live module when the reference
    tree is present (the same comparison, recomputed)."""
    from oracle import s1_oracle as S1
    g, meta = load_golden("s1_tiny_decode.npz")
    cfg = S1.S1Config.from_dict(meta["config"])
    P = S1.make_params(cfg, seed=meta["seed"])
    ct, cb = torch.from_numpy(g["code_t"]), torch.from_numpy(g["code_b"])
    px = S1.decode_code(P, cfg, ct, cb)
    assert tuple(px.shape) == (ct.shape[0], 3, cfg.resolution, cfg.resolution)
    assert float((px - torch.from_numpy(g["pixels"])).abs().max()) < 1e-5
    if R.reference_available():
        model = R.build_reference_stage1(cfg, P)
        with torch.no_grad():
            want = model.decode_code(ct, cb)
        assert float((px - want).abs().max()) < 1e-5


def test_oracle_3level_equals_reference_golden_and_live_reference():
    """SURVEY.md 8f-2: oracle/hq3_oracle.py against the grids of the unmodified 3-level HQTransformer ('parallel-add')."""
    from oracle import hq3_oracle as O3
    g, meta = load_golden("tiny3_cls_greedy.npz")
    cfg = O3.HQ3Config.from_dict(meta["config"])
    assert meta["min_logit_margin"] >= 1e-4
    P = O3.make_params(cfg, seed=meta["seed"])
    labels = torch.from_numpy(g["labels"])
    S = g["codes_top"].shape[1]
    ct, cm, cb = O3.sample(P, cfg, labels, len(labels), top_k=(1, 1, 1), max_seq_len=S)
    assert np.array_equal(ct.numpy(), g["codes_top"]) and np.array_equal(cm.numpy(), g["codes_mid"])
    assert np.array_equal(cb.numpy(), g["codes_bot"])
    # stochastic 3-level run with per-level top-k / top-p / temperatures under a fixed torch seed
    _check_seeded_runs("tiny3_cls_stochastic.npz")
