"""-m gpu: image completion (hq_run_args.prefix_len, `sampling_ihqgpt(prefix_code_top=, prefix_code_bot=)`,
`sampling_hqtransformer(prefix_codes=)`): positions < P are given, their spatial KV cache comes from one causal pass over the
prefix, positions >= P are sampled by the ordinary loop.

- the prefix attention kernel against fp64 at every query / key count 1..127;
- greedy completions of the reference-made goldens (fp32 engine) reproduce the golden grids bit for bit;
- logits at positions >= P against the oracle (fp32 / bf16-emulating / fp16-emulating) within the bars of the existing
  logit tests, and against the existing forced loop (given codes through every position) at B up to 300;
- launch-mode invariance, determinism, batch cuts, shared prefix, graph keys per P, validation, workspace accounting."""
from dataclasses import replace

import numpy as np
import pytest
import torch

from hqtransformer_b200 import engine as E
from oracle import hq_oracle as O
from oracle import hq3_oracle as O3
from tests import fp16_emulation as F
from tests.helpers import build_model, cfg_from_meta, load_golden
from tests.test_gpu_level3 import _model as _model3

pytestmark = pytest.mark.gpu

GREEDY = dict(top_k_top=1, top_p_top=1.0, top_k_bot=1, top_p_bot=1.0, softmax_temperature=[1.0, 1.0])
STOCH = dict(top_k_top=50, top_p_top=0.9, top_k_bot=50, top_p_bot=0.9, softmax_temperature=[0.9, 0.9])
GOLDENS = ["tiny_cls_greedy.npz", "small_cls_greedy.npz", "asym_cls_greedy.npz", "tiny_txt_greedy.npz", "asym_txt_greedy.npz",
           "tiny_reduce_uncond_greedy.npz", "tiny_pos2d_cls_greedy.npz", "tiny_top2bot_cls_greedy.npz",
           "tiny_bidir_cls_greedy.npz", "asym_top2bot_reduce_pos2d_greedy.npz", "l12_cls_greedy_b4.npz"]
# logit bars of the existing tests: fp32 vs reference (test_step_logits_fp32_vs_reference), bf16 vs the bf16-emulating
# oracle (test_step_logits_bf16_vs_oracle_and_reference), fp16 vs the fp16-emulating oracle (test_gpu_fp16.py)
BARS = {"fp32": (2e-5, 2e-5), "bf16": (2e-2, 2e-3), "fp16": (4e-3, 5e-4)}


def _golden(name):
    g, meta = load_golden(name)
    cfg = cfg_from_meta(meta)
    cond = (torch.from_numpy(g["text_ids"]) if cfg.cond == "txt" else
            torch.from_numpy(g["labels"]) if cfg.cond == "cls" else None)
    return g, meta, cfg, cond


# ------------------------------------------------------------------------------------------------
# the prefix attention kernel
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16, torch.float32], ids=["bf16", "fp16", "fp32"])
def test_prefix_attention_vs_fp64_every_length(dtype):
    """hq_debug_attention_prefix at n_q = 1..127 (query i over keys 0..i) against fp64 causal softmax attention of the same
    2-byte / fp32 operands.  Bar: the output type's unit roundoff (2^-8 bf16, 2^-11 fp16) relative plus 1e-4 (the head /
    tail split carries P to ~2^-17; fp32 accumulation); fp32: 2e-6.  Keys past n_q in the cache are NaN and must not reach the output; repeated launches
    give the same bits."""
    B, T, nh = 3, 128, 3
    D = nh * 64
    g = torch.Generator(device="cuda").manual_seed(11)
    q = (torch.randn(B, T, D, generator=g, device="cuda") * 2).to(dtype)
    K = (torch.randn(B, T, D, generator=g, device="cuda") * 2).to(dtype)
    V = torch.randn(B, T, D, generator=g, device="cuda").to(dtype)
    unit = {torch.bfloat16: 2.0 ** -8, torch.float16: 2.0 ** -11, torch.float32: 0.0}[dtype]
    worst = 0.0
    for n_q in range(1, 128):
        Kn, Vn = K.clone(), V.clone()
        Kn[:, n_q:] = float("nan")
        Vn[:, n_q:] = float("nan")
        qn = q[:, :n_q].contiguous()
        got = E.debug_attention_prefix(qn, Kn, Vn)
        qh = qn.double().view(B, n_q, nh, 64)
        Kh = K.double()[:, :n_q].view(B, n_q, nh, 64)
        Vh = V.double()[:, :n_q].view(B, n_q, nh, 64)
        s = torch.einsum("bihd,bjhd->bhij", qh, Kh) / 8.0
        mask = torch.ones(n_q, n_q, dtype=torch.bool, device="cuda").tril()
        s = s.masked_fill(~mask, float("-inf"))
        ref = torch.einsum("bhij,bjhd->bihd", torch.softmax(s, -1), Vh).reshape(B, n_q, D)
        err = (got.double() - ref).abs()
        bar = unit * ref.abs() + (1e-4 if unit else 2e-6)
        assert bool(torch.isfinite(got.double()).all()), f"n_q={n_q}: non-finite output"
        assert bool((err <= bar).all()), f"n_q={n_q}: max err {err.max():.3e}"
        worst = max(worst, float(err.max()))
        assert torch.equal(got, E.debug_attention_prefix(qn, Kn, Vn)), f"n_q={n_q}: repeated launch differs"
    print(f"{dtype}: prefix attention max err over n_q 1..127: {worst:.3e}")


# ------------------------------------------------------------------------------------------------
# completions of the reference goldens (fp32 engine, greedy): bit for bit
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", GOLDENS)
def test_greedy_completion_reproduces_reference_golden(name):
    import hqtransformer_b200 as H
    g, meta, cfg, cond = _golden(name)
    P_ = O.make_params(cfg, seed=meta["seed"], init=meta["init"])
    ct_g, cb_g = torch.from_numpy(g["codes_top"]), torch.from_numpy(g["codes_bot"])
    B, S = ct_g.shape
    model = build_model(cfg, P_, precision="fp32", max_batch=B, max_seq_len=S)
    for P in (1, 17, S - 1):
        pt, pb = ct_g[:, :P].clone(), cb_g[:, :P].clone()
        ct, cb = H.sampling_ihqgpt(model, B, cond, use_fp16=False, max_seq_len=S, is_tqdm=False, prefix_code_top=pt,
                                   prefix_code_bot=pb, **GREEDY)
        assert torch.equal(ct[:, :P].cpu(), pt) and torch.equal(cb[:, :P].cpu(), pb), f"P={P}: prefix changed"
        assert np.array_equal(ct.cpu().numpy(), g["codes_top"]), f"P={P}: top codes differ from the golden"
        assert np.array_equal(cb.cpu().numpy(), g["codes_bot"]), f"P={P}: bottom codes differ from the golden"


def test_greedy_completion_reproduces_level3_golden():
    import hqtransformer_b200 as H
    g, meta = load_golden("tiny3_cls_greedy.npz")
    cfg = O3.HQ3Config.from_dict(meta["config"])
    P_ = O3.make_params(cfg, seed=meta["seed"])
    labels = torch.from_numpy(g["labels"])
    want = [torch.from_numpy(g[k]) for k in ("codes_top", "codes_mid", "codes_bot")]
    B, S = want[0].shape
    m = _model3(cfg, P_, "fp32", B, max_seq_len=S)
    for P in (1, 17, S - 1):
        got = H.sampling_hqtransformer(m, B, labels, top_k=[1, 1, 1], top_p=[1.0, 1.0, 1.0], use_fp16=False, max_seq_len=S,
                                       is_tqdm=False, prefix_codes=[w[:, :P] for w in want])
        for a, b in zip(got, want):
            assert torch.equal(a.cpu(), b), f"P={P}: 3-level completion differs from the golden"


# ------------------------------------------------------------------------------------------------
# logits at positions >= P
# ------------------------------------------------------------------------------------------------
def _completion_logits(model, prec, cond, ct, cb, P, fill=7.0):
    """Teacher-forced logits of a completion: prefix = ct / cb[:, :P], given_top / given_bot = ct / cb (positions >= P).
    Rows of positions < P start as `fill`, the rest as 0 (what step_logits and the oracles leave in unused columns)."""
    B, S = ct.shape
    eng = model.engine(prec)
    if B > eng.max_batch:
        eng.reserve_batch(B)
    cond_t = model.build_sos(cond, B)
    dev = model.device
    ct_d, cb_d = ct.to(dev).contiguous(), cb.to(dev).contiguous()
    logits = torch.zeros(B, S, 5, eng.vocab_max, dtype=torch.float32, device=dev)
    logits[:, :P] = fill
    eng.run(batch=B, seq_len=S, pos_begin=0, pos_end=S, sampling=E.SamplingParams(), cond=cond_t, given_top=ct_d, given_bot=cb_d,
            codes_top=ct_d.clone(), codes_bot=cb_d.clone(), logits=logits, prefix_len=P)
    return logits.cpu()


def _check(what, got, want, prec):
    mx, mean = BARS[prec]
    d = (got - want).abs()
    print(f"{what}: max {d.max():.3e} mean {d.mean():.3e}")
    assert float(d.max()) <= mx and float(d.mean()) <= mean, (what, float(d.max()), float(d.mean()))


@pytest.mark.parametrize("prec", ["fp32", "bf16", "fp16"])
@pytest.mark.parametrize("name", ["small_cls_greedy.npz", "asym_txt_greedy.npz", "tiny_bidir_cls_greedy.npz"])
def test_completion_logits_vs_oracle(name, prec):
    """fp32 against the reference-rounded fp32 oracle, bf16 against the bf16-emulating oracle, fp16 against the
    fp16-emulating oracle; the caller's logits rows of positions < P are left as they were."""
    g, meta, cfg, cond = _golden(name)
    P_ = O.make_params(cfg, seed=meta["seed"], init=meta["init"])
    ct, cb = torch.from_numpy(g["codes_top"]), torch.from_numpy(g["codes_bot"])
    B, S = ct.shape
    model = build_model(cfg, P_, precision=prec, max_batch=B, max_seq_len=S)
    if prec == "fp32":
        ref = O.step_logits(P_, cfg, cond, ct, cb)
    elif prec == "bf16":
        ref = O.step_logits(P_, cfg, cond, ct, cb, emulate="bf16")
    else:
        ref = F.step_logits(P_, cfg, cond, ct, cb)
    V = ref.shape[-1]
    for P in (1, 17, S - 1):
        lg = _completion_logits(model, prec, cond, ct, cb, P)
        assert bool((lg[:, :P] == 7.0).all()), f"P={P}: logits of prefix positions were written"
        _check(f"{name} {prec} P={P} vs oracle", lg[:, P:, :, :V], ref[:, P:], prec)


@pytest.mark.parametrize("prec", ["fp32", "bf16", "fp16"])
@pytest.mark.parametrize("kw,B", [(dict(), 300), (dict(cond="txt"), 130), (dict(model_type="top2bot"), 140),
                                  (dict(model_type="bidirectional", embedding_type="reduce", position_embedding="2d"), 150)])
def test_prefill_path_equals_forced_loop(kw, B, prec):
    """The same completion through the prefix pass and through the existing forced loop (given codes at every position,
    step_logits): logits at positions >= P agree within the bars above, at B up to 300 (CTA-pair GEMMs in both paths)."""
    import hqtransformer_b200 as H
    cfg = replace(O.ASYM if kw.get("cond") == "txt" else O.SMALL, **kw)
    P_ = O.make_params(cfg, seed=4, init="rich")
    S = 12
    g = torch.Generator().manual_seed(B)
    cond = (torch.randint(0, cfg.vocab_txt, (B, cfg.ctx_len_txt), generator=g) if cfg.cond == "txt" else
            torch.randint(0, cfg.n_classes, (B,), generator=g))
    ct = torch.randint(0, cfg.vocab_top, (B, S), generator=g)
    cb = torch.randint(0, cfg.vocab_bot, (B, S, 4), generator=g)
    model = build_model(cfg, P_, precision=prec, max_batch=B, max_seq_len=S)
    forced = H.step_logits(model, cond, ct, cb, use_fp16=prec != "fp32").cpu()
    for P in (1, 5, S - 1):
        lg = _completion_logits(model, prec, cond, ct, cb, P)
        _check(f"{kw} B={B} {prec} P={P}: prefill vs forced loop", lg[:, P:], forced[:, P:], prec)


def test_level3_completion_logits_vs_oracle():
    import hqtransformer_b200 as H  # noqa: F401
    cfg = O3.SMALL3
    P_ = O3.make_params(cfg, seed=7)
    B, S = 20, 5
    g = torch.Generator().manual_seed(2)
    labels = torch.randint(0, cfg.n_classes, (B,), generator=g)
    given = torch.stack([torch.randint(0, cfg.vocab_sizes[0 if j == 0 else (1 if j < 5 else 2)], (B, S), generator=g)
                         for j in range(21)], dim=-1)
    codes = [given[:, :, 0].contiguous(), given[:, :, 1:5].contiguous(), given[:, :, 5:].contiguous()]
    for prec in ("fp32", "bf16", "fp16"):
        if prec == "fp16":
            _, ref = F.sample3(P_, cfg, labels, B, max_seq_len=S, given=given, return_logits=True)
        else:
            _, ref = O3.sample(P_, cfg, labels, B, max_seq_len=S, given=given, return_logits=True,
                               **({"emulate": "bf16"} if prec == "bf16" else {}))
        m = _model3(cfg, P_, prec, B, max_seq_len=S)
        eng = m.engine(prec)
        dev = m.device
        for P in (1, 3):
            c = [t.to(dev) for t in codes]
            logits = torch.zeros(B, S, 21, eng.vocab_max, device=dev)
            logits[:, :P] = 7.0
            eng.run(batch=B, seq_len=S, pos_begin=0, pos_end=S, sampling=E.SamplingParams(), cond=m.build_cond(labels, B),
                    given_top=c[0], given_mid=c[1], given_bot=c[2], codes_top=c[0].clone(), codes_mid=c[1].clone(),
                    codes_bot=c[2].clone(), logits=logits, prefix_len=P)
            lg = logits.cpu()
            assert bool((lg[:, :P] == 7.0).all())
            _check(f"3-level {prec} P={P} vs oracle", lg[:, P:, :, :ref.shape[-1]], ref[:, P:], prec)


# ------------------------------------------------------------------------------------------------
# invariances
# ------------------------------------------------------------------------------------------------
def _small(prec, B, S=16, **kw):
    cfg = O.SMALL
    P_ = O.make_params(cfg, seed=5, init="rich")
    return cfg, build_model(cfg, P_, precision=prec, max_batch=B, max_seq_len=S, **kw)


def _prefix(cfg, B, P, seed=0):
    g = torch.Generator().manual_seed(seed)
    return torch.randint(0, cfg.vocab_top, (B, P), generator=g), torch.randint(0, cfg.vocab_bot, (B, P, 4), generator=g)


@pytest.mark.parametrize("prec", ["bf16", "fp16", "fp32"])
def test_graph_pdl_equals_stream_launches_and_deterministic(prec):
    import hqtransformer_b200 as H
    B, S = 300 if prec != "fp32" else 40, 16
    cfg, base = _small(prec, B, S, use_cuda_graph=False, use_pdl=False)
    _, model = _small(prec, B, S, use_cuda_graph=True, use_pdl=True)
    labels = torch.arange(B) % cfg.n_classes
    pt, pb = _prefix(cfg, B, 6)
    kw = dict(use_fp16=prec != "fp32", max_seq_len=S, is_tqdm=False, seed=7, prefix_code_top=pt, prefix_code_bot=pb, **STOCH)
    ct0, cb0 = H.sampling_ihqgpt(base, B, labels, **kw)
    for _ in range(3):
        ct, cb = H.sampling_ihqgpt(model, B, labels, **kw)
        assert torch.equal(ct, ct0) and torch.equal(cb, cb0)


@pytest.mark.parametrize("cuts", [(0, 19, 37), (0, 1, 36, 37), (0, 150, 300)])
def test_completion_does_not_depend_on_how_the_batch_is_cut(cuts):
    import hqtransformer_b200 as H
    B, S = cuts[-1], 16
    cfg, model = _small("bf16", B, S)
    labels = torch.randint(0, cfg.n_classes, (B,), generator=torch.Generator().manual_seed(0))
    pt, pb = _prefix(cfg, B, 9, seed=1)
    for kw in (dict(top_k_top=1, top_k_bot=1), STOCH):
        ct, cb = H.sampling_ihqgpt(model, B, labels, max_seq_len=S, is_tqdm=False, seed=3, prefix_code_top=pt,
                                   prefix_code_bot=pb, **kw)
        for lo, hi in zip(cuts[:-1], cuts[1:]):
            ct_s, cb_s = H.sampling_ihqgpt(model, hi - lo, labels[lo:hi], max_seq_len=S, is_tqdm=False, seed=3, row_offset=lo,
                                           prefix_code_top=pt[lo:hi], prefix_code_bot=pb[lo:hi], **kw)
            assert torch.equal(ct_s, ct[lo:hi]) and torch.equal(cb_s, cb[lo:hi]), (lo, hi, kw)


@pytest.mark.parametrize("prec", ["bf16", "fp16", "fp32"])
@pytest.mark.parametrize("variant", ["cls", "txt", "bidirectional", "level3"])
def test_shared_prefix_equals_per_row_prefix(variant, prec):
    """One condition and one prefix for every row: the prefix pass for row 0 plus the broadcast gives the same grids as the
    per-row prefix pass (and the auto-detection picks the shared form)."""
    import hqtransformer_b200 as H
    B, S, P = 7, 8, 5
    if variant == "level3":
        cfg = O3.TINY3
        P_ = O3.make_params(cfg, seed=3)
        m = _model3(cfg, P_, prec, B, max_seq_len=S)
        g = torch.Generator().manual_seed(4)
        pre = [torch.randint(0, cfg.vocab_sizes[0], (1, P), generator=g), torch.randint(0, cfg.vocab_sizes[1], (1, P, 4), generator=g),
               torch.randint(0, cfg.vocab_sizes[2], (1, P, 16), generator=g)]
        kw = dict(top_k=[20, 20, 20], use_fp16=prec != "fp32", max_seq_len=S, is_tqdm=False, seed=5, prefix_codes=pre)
        a = H.sampling_hqtransformer(m, B, 3, shared_prefix=False, **kw)
        b = H.sampling_hqtransformer(m, B, 3, shared_prefix=True, **kw)
        c = H.sampling_hqtransformer(m, B, 3, **kw)
        for x, y, z in zip(a, b, c):
            assert torch.equal(x, y) and torch.equal(x, z)
            assert torch.equal(x[:1].expand_as(x)[:, :P], x[:, :P])
        return
    cfg = replace(O.ASYM, cond="txt") if variant == "txt" else replace(O.TINY, model_type=variant) if variant != "cls" else O.TINY
    P_ = O.make_params(cfg, seed=6, init="rich")
    model = build_model(cfg, P_, precision=prec, max_batch=B, max_seq_len=S)
    cond = (torch.randint(0, cfg.vocab_txt, (1, cfg.ctx_len_txt), generator=torch.Generator().manual_seed(3)).repeat(B, 1)
            if variant == "txt" else 4)
    pt, pb = _prefix(cfg, 1, P, seed=2)
    for kw in (dict(top_k_top=1, top_k_bot=1), dict(top_k_top=20, top_k_bot=30, softmax_temperature=[0.9, 1.1])):
        kw.update(max_seq_len=S, is_tqdm=False, use_fp16=prec != "fp32", seed=5, prefix_code_top=pt, prefix_code_bot=pb)
        a = H.sampling_ihqgpt(model, B, cond, shared_prefix=False, **kw)
        b = H.sampling_ihqgpt(model, B, cond, shared_prefix=True, **kw)
        c = H.sampling_ihqgpt(model, B, cond, **kw)
        assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
        assert torch.equal(a[0], c[0]) and torch.equal(a[1], c[1])
        assert bool((a[0][:, :P].cpu() == pt).all()) and bool((a[1][:, :P].cpu() == pb).all())


def test_switching_prefix_length_never_replays_a_stale_graph():
    """P = 5, 9, 5, 0, 12, 9 on one graph-replaying context, each against a fresh context with plain stream launches."""
    import hqtransformer_b200 as H
    B, S = 9, 16
    cfg, model = _small("bf16", B, S)
    _, plain = _small("bf16", B, S, use_cuda_graph=False, use_pdl=False)
    labels = torch.arange(B) % cfg.n_classes
    for P in (5, 9, 5, 0, 12, 9):
        kw = dict(max_seq_len=S, is_tqdm=False, seed=11, **STOCH)
        if P:
            pt, pb = _prefix(cfg, B, P, seed=P)
            kw.update(prefix_code_top=pt, prefix_code_bot=pb)
        ct, cb = H.sampling_ihqgpt(model, B, labels, **kw)
        ct0, cb0 = H.sampling_ihqgpt(plain, B, labels, **kw)
        assert torch.equal(ct, ct0) and torch.equal(cb, cb0), f"P={P}"


def test_given_codes_apply_after_the_prefix_only():
    import hqtransformer_b200 as H
    B, S, P = 4, 10, 6
    cfg, model = _small("fp32", B, S)
    pt, pb = _prefix(cfg, B, P, seed=8)
    given = torch.randint(0, cfg.vocab_top, (B, S), generator=torch.Generator().manual_seed(9))
    ct, cb = H.sampling_ihqgpt(model, B, 2, use_fp16=False, max_seq_len=S, is_tqdm=False, seed=1, given_top_code=given,
                               prefix_code_top=pt, prefix_code_bot=pb)
    assert torch.equal(ct[:, :P].cpu(), pt) and torch.equal(cb[:, :P].cpu(), pb)
    assert torch.equal(ct[:, P:].cpu(), given[:, P:])


def test_completion_of_own_prefix_with_own_seed_redraws_the_stream():
    """Same Philox counters: completing a sampled grid's prefix with its seed gives back (nearly) the same tail - exactly,
    unless a last-bit logit difference between the prefix pass and the step path moves one draw across a CDF boundary."""
    import hqtransformer_b200 as H
    B, S = 16, 32
    cfg, model = _small("fp32", B, S)
    labels = torch.arange(B) % cfg.n_classes
    kw = dict(use_fp16=False, max_seq_len=S, is_tqdm=False, seed=21, **STOCH)
    ct, cb = H.sampling_ihqgpt(model, B, labels, **kw)
    P = 12
    ct2, cb2 = H.sampling_ihqgpt(model, B, labels, prefix_code_top=ct[:, :P], prefix_code_bot=cb[:, :P], **kw)
    agree = float((ct2[:, P:] == ct[:, P:]).float().mean())
    print(f"fp32 completion of the own prefix: {agree:.4f} of the top codes at >= P agree")
    assert agree >= 0.9


# ------------------------------------------------------------------------------------------------
# validation and workspace
# ------------------------------------------------------------------------------------------------
def test_c_abi_validation_errors():
    B, S = 2, 8
    cfg, model = _small("bf16", B, S)
    eng = model.engine("bf16")
    dev = model.device
    ct = torch.zeros(B, S, dtype=torch.int64, device=dev)
    cb = torch.zeros(B, S, 4, dtype=torch.int64, device=dev)
    cond = torch.zeros(B, dtype=torch.int64, device=dev)
    base = dict(batch=B, seq_len=S, sampling=E.SamplingParams(), cond=cond, codes_top=ct, codes_bot=cb)
    for kw, msg in ((dict(pos_begin=0, pos_end=S, prefix_len=-1), "prefix_len must be >= 0"),
                    (dict(pos_begin=1, pos_end=S, prefix_len=2), "needs pos_begin == 0"),
                    (dict(pos_begin=0, pos_end=4, prefix_len=4), "must be below pos_end"),
                    (dict(pos_begin=0, pos_end=4, prefix_len=7), "must be below pos_end")):
        with pytest.raises(E._lib.HQError, match=msg):
            eng.run(**base, **kw)
    # a completion leaves the ctx usable
    eng.run(**base, pos_begin=0, pos_end=S, prefix_len=3)


def test_longest_text_prefix_fits_the_attention_keys():
    """A 60-token prompt and P = 63 of 64 positions: 122 prefix tokens in one pass (hq_create already bounds T0 + S - 1 by
    the 128 keys, so validate_run's own bound on T0 + P - 1 never fires for a ctx that exists)."""
    import hqtransformer_b200 as H
    cfg = replace(O.TINY, cond="txt", ctx_len_txt=60, ctx_len_img=64)
    P_ = O.make_params(cfg, seed=1, init="rich")
    model = build_model(cfg, P_, precision="bf16", max_batch=2, max_seq_len=64)
    ids = torch.randint(0, cfg.vocab_txt, (2, 60), generator=torch.Generator().manual_seed(0))
    pt, pb = _prefix(cfg, 2, 63)
    ct, cb = H.sampling_ihqgpt(model, 2, ids, max_seq_len=64, is_tqdm=False, seed=1, prefix_code_top=pt, prefix_code_bot=pb)
    assert torch.equal(ct[:, :63].cpu(), pt) and int(ct.max()) < cfg.vocab_top


def test_python_validation_errors():
    import hqtransformer_b200 as H
    B, S = 3, 8
    cfg, model = _small("bf16", B, S)
    pt, pb = _prefix(cfg, B, 4)
    run = lambda **kw: H.sampling_ihqgpt(model, B, 1, max_seq_len=S, is_tqdm=False, **kw)  # noqa: E731
    with pytest.raises(ValueError, match="go together"):
        run(prefix_code_top=pt)
    with pytest.raises(ValueError, match="must be"):
        run(prefix_code_top=pt[:, :, None], prefix_code_bot=pb)
    with pytest.raises(ValueError, match="must be"):
        run(prefix_code_top=pt[:2], prefix_code_bot=pb[:2])
    with pytest.raises(ValueError, match="positions"):
        run(prefix_code_top=pt, prefix_code_bot=pb[:, :3])
    with pytest.raises(ValueError, match="outside"):
        run(prefix_code_top=torch.zeros(B, S, dtype=torch.int64), prefix_code_bot=torch.zeros(B, S, 4, dtype=torch.int64))
    with pytest.raises(IndexError):
        run(prefix_code_top=pt + cfg.vocab_top, prefix_code_bot=pb)
    with pytest.raises(ValueError, match="integer"):
        run(prefix_code_top=pt.float(), prefix_code_bot=pb)


def test_workspace_growth_is_counted_and_prefix_free_runs_allocate_nothing():
    import hqtransformer_b200 as H
    B, S = 6, 16
    cfg, model = _small("bf16", B, S)
    eng = model.engine("bf16")
    labels = torch.arange(B) % cfg.n_classes
    kw = dict(max_seq_len=S, is_tqdm=False, seed=1)
    base = eng.device_bytes
    H.sampling_ihqgpt(model, B, labels, **kw)
    assert eng.device_bytes == base, "a run without a prefix allocated device memory"
    sizes = []
    for P in (4, 3, 9, 9, 2):
        pt, pb = _prefix(cfg, B, P)
        H.sampling_ihqgpt(model, B, labels, prefix_code_top=pt, prefix_code_bot=pb, **kw)
        sizes.append(eng.device_bytes)
    assert sizes[0] > base and sizes[1] == sizes[0] and sizes[2] > sizes[1] and sizes[3] == sizes[2] == sizes[4], sizes
    H.sampling_ihqgpt(model, B, labels, **kw)
    assert eng.device_bytes == sizes[-1]
    eng.reserve_batch(B)
    assert eng.device_bytes == base, "hq_reserve_batch kept the prefix workspace"
