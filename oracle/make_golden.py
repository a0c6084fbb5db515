"""TEST INFRASTRUCTURE ONLY - generates tests/golden/*.npz by running the UNMODIFIED reference.

Run in the build container (where /root/reference exists):

    python -m oracle.make_golden            # writes tests/golden/ (small models + filters)
    python -m oracle.make_golden --full-size    # only the ImageNet-L12-size golden (BASELINE config 1 at real scale)
    python -m oracle.make_golden --level3       # only the 3-level HQTransformer golden
    python -m oracle.make_golden --stage1       # only the stage-1 decode golden (SimRQGAN2Generator.decode_code)
    python -m oracle.make_golden --variants     # only the 8f-3 model variants (reduce / 2d / top2bot / bidirectional)
    python -m oracle.make_golden --all
    python -m oracle.make_golden --live-checks  # only the seeded runs the tests also repeat against the live reference
                                                # (written from the oracle; re-checked against the reference when present)

The reference has no tests or golden vectors of its own (SURVEY.md section 4), so these files are the
pinned known answers for the hot path: they are produced by the reference's own code
(`sampling_ihqgpt`, `iHQGPT.sampling_step`, `cutoff_topk_logits`, `cutoff_topp_probs`) on CPU, fp32,
on weights that `oracle.hq_oracle.make_params(cfg, seed, init)` regenerates deterministically (same
torch build on the GPU box), so only the tiny outputs are committed.
"""
from __future__ import annotations

import json
import os
import sys

import numpy as np
import torch

from oracle import hq_oracle as O
from oracle import ref_shim as R

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")
LOGIT_POSITIONS = [0, 1, 2, 31, 63]


def reference_sample_rows(model, sos, max_seq_len, capture=None, **kw):
    """The 40-line outer loop of sampling.py:178-237 re-driven here so that every row can carry its
    own class (`sos = model.sos(labels).unsqueeze(1)`); each position calls the reference's
    `iHQGPT.sampling_step` unchanged."""
    codes_top = codes_bot = past = None
    B = sos.shape[0]
    for cnt in range(max_seq_len):
        if codes_top is None:
            ct = cb = pos = None
        else:
            ct = codes_top[:, cnt - 1:cnt]
            cb = codes_bot[:, cnt - 1, :]
            pos = torch.full((B, 1), cnt - 1, dtype=torch.long)
        if capture is not None:
            capture["cnt"] = cnt
        code_top, code_bot, present = model.sampling_step(sos=sos, codes_t=ct, codes_b=cb, pos_codes=pos,
                                                          use_fp16=False, past=past, **kw)
        present = torch.stack(present).clone()
        past = [present] if past is None else past + [present]
        codes_top = code_top if codes_top is None else torch.cat([codes_top, code_top], 1)
        codes_bot = code_bot if codes_bot is None else torch.cat([codes_bot, code_bot], 1)
    return codes_top, codes_bot


def run_with_logit_capture(model, sos, max_seq_len, positions=None, **kw):
    cap = {"cnt": 0, "top": {}, "bot": {}}
    h1 = model.head_top.register_forward_hook(
        lambda m, i, o: cap["top"].__setitem__(cap["cnt"], o.detach().clone().reshape(o.shape[0], -1)))
    h2 = model.head_bot.register_forward_hook(
        lambda m, i, o: cap["bot"].__setitem__(cap["cnt"], o.detach().clone()))
    try:
        ct, cb = reference_sample_rows(model, sos, max_seq_len, capture=cap, **kw)
    finally:
        h1.remove()
        h2.remove()
    lg = []
    for p in (LOGIT_POSITIONS if positions is None else positions):
        if p < max_seq_len:
            top, bot = cap["top"][p], cap["bot"][p]                                     # [B,Vt], [B,4,Vb]
            V = max(top.shape[-1], bot.shape[-1])                                       # zero-padded like O.sample
            row = torch.zeros(top.shape[0], 5, V)
            row[:, 0, : top.shape[-1]] = top
            row[:, 1:, : bot.shape[-1]] = bot
            lg.append(row)                                                              # [B,5,V]
    return ct, cb, torch.stack(lg, dim=1)                                               # [B,P,5,V]


def min_margin(logits):
    top2 = torch.topk(logits, 2, dim=-1).values
    return float((top2[..., 0] - top2[..., 1]).min())


def full_run_margin(cfg, P, cond, B):
    """Smallest top-1/top-2 logit gap over ALL 320*B greedy decisions of the run (computed with the
    oracle, which is bit-identical to the reference on CPU).  The seeds below were picked so that this
    margin is >= 1e-4: an fp32 GPU run (different summation order, ~1e-6 error) then cannot flip an
    argmax, which is what makes 'bit-exact greedy code grids' a meaningful assertion."""
    _, _, lg = O.sample(P, cfg, cond, B, top_k_top=1, top_k_bot=1, return_logits=True)
    return min(min_margin(lg[:, :, 0, : cfg.vocab_top]), min_margin(lg[:, :, 1:, : cfg.vocab_bot]))


def meta(cfg, seed, init, **extra):
    d = dict(config=cfg.to_dict(), seed=seed, init=init, torch=torch.__version__,
             reference="kakaobrain/hqtransformer (read-only tree at /root/reference)")
    d.update(extra)
    return np.array(json.dumps(d))


GREEDY = dict(top_k_top=1, top_p_top=1.0, top_k_bot=1, top_p_bot=1.0, softmax_temperature=[1.0, 1.0])


def golden_cls(cfg, name, seed, init, labels):
    P = O.make_params(cfg, seed=seed, init=init)
    model = R.build_reference_model(cfg, P)
    labels_t = torch.tensor(labels, dtype=torch.long)
    sos = model.sos(labels_t).unsqueeze(1)
    ct, cb, lg = run_with_logit_capture(model, sos, 64, **GREEDY)
    # the reference's own driver: one scalar class for the whole batch (sampling.py:183-186)
    ct_s, cb_s = R.reference_sample(model, len(labels), int(labels[-1]), max_seq_len=64, **GREEDY)
    assert torch.equal(ct_s[0], ct[-1]) and torch.equal(cb_s[0], cb[-1])
    np.savez_compressed(os.path.join(GOLDEN_DIR, name),
                        meta=meta(cfg, seed, init, labels=list(labels), logit_positions=LOGIT_POSITIONS,
                                  min_logit_margin=full_run_margin(cfg, P, labels_t, len(labels))),
                        labels=np.asarray(labels, dtype=np.int64),
                        codes_top=ct.numpy(), codes_bot=cb.numpy(),
                        codes_top_scalar_class=ct_s.numpy(), codes_bot_scalar_class=cb_s.numpy(),
                        logits=lg.numpy().astype(np.float32))
    print(name, "min greedy margin over the run", full_run_margin(cfg, P, labels_t, len(labels)))


def golden_cls_full_size(cfg, name, seed, labels, logit_positions=(63,)):
    """BASELINE config 1 at the reference's REAL scale (ImageNet L12: D=1536, 12+4 layers, V=8192, 530 M parameters,
    `_init_weights` statistics): batch 4 with per-row classes, greedy, all 64 positions, fp32 on CPU through the
    reference's own `iHQGPT.sampling_step`.  Only the code grids and the head outputs at `logit_positions` are stored;
    the weights are regenerated from (cfg, seed) by `make_params`."""
    P = O.make_params(cfg, seed=seed, init="reference")
    model = R.build_reference_model(cfg, P)
    labels_t = torch.tensor(labels, dtype=torch.long)
    sos = model.sos(labels_t).unsqueeze(1)
    ct, cb, lg = run_with_logit_capture(model, sos, 64, positions=list(logit_positions), **GREEDY)
    margin = full_run_margin(cfg, P, labels_t, len(labels))
    np.savez_compressed(os.path.join(GOLDEN_DIR, name),
                        meta=meta(cfg, seed, "reference", labels=list(labels), logit_positions=list(logit_positions),
                                  min_logit_margin=margin),
                        labels=np.asarray(labels, dtype=np.int64), codes_top=ct.numpy(), codes_bot=cb.numpy(),
                        logits=lg.numpy().astype(np.float32))
    print(name, "min greedy margin over the run", margin)


def golden_txt(cfg, name, seed, init, B):
    P = O.make_params(cfg, seed=seed, init=init)
    model = R.build_reference_model(cfg, P)
    g = torch.Generator().manual_seed(seed + 1000)
    ids = torch.randint(0, cfg.vocab_txt, (B, cfg.ctx_len_txt), generator=g)
    ct, cb = R.reference_sample(model, 1, ids, max_seq_len=64, **GREEDY)
    np.savez_compressed(os.path.join(GOLDEN_DIR, name),
                        meta=meta(cfg, seed, init, min_logit_margin=full_run_margin(cfg, P, ids, B)),
                        text_ids=ids.numpy(), codes_top=ct.numpy(), codes_bot=cb.numpy())
    print(name, "done")


def golden_uncond(cfg, name, seed, init, B):
    P = O.make_params(cfg, seed=seed, init=init)
    model = R.build_reference_model(cfg, P)
    torch.manual_seed(seed + 7)
    kw = dict(top_k_top=8, top_p_top=0.9, top_k_bot=16, top_p_bot=0.95, softmax_temperature=[0.9, 1.1])
    ct, cb = R.reference_sample(model, B, None, max_seq_len=64, **kw)     # stochastic, global torch RNG
    np.savez_compressed(os.path.join(GOLDEN_DIR, name), meta=meta(cfg, seed, init, torch_seed=seed + 7, **kw),
                        codes_top=ct.numpy(), codes_bot=cb.numpy())
    print(name, "done")


def golden_variant(cfg, name, seed, init, labels=None, B=3):
    """SURVEY.md 8f-3 variants of the 2-level model (embedding_type 'reduce', position_embedding '2d', model_type 'top2bot' /
    'bidirectional', unconditional sos): greedy code grids of the reference's own sampler; class-conditional models are
    driven row by row with per-row classes (`iHQGPT.sampling_step` unchanged), unconditional ones through `sampling_ihqgpt`."""
    P = O.make_params(cfg, seed=seed, init=init)
    model = R.build_reference_model(cfg, P)
    if cfg.cond == "cls":
        labels_t = torch.tensor(labels, dtype=torch.long)
        ct, cb = reference_sample_rows(model, model.sos(labels_t).unsqueeze(1), 64, **GREEDY)
        cond, n = labels_t, len(labels)
        extra = dict(labels=np.asarray(labels, dtype=np.int64))
    else:
        ct, cb = R.reference_sample(model, B, None, max_seq_len=64, **GREEDY)
        cond, n = None, B
        extra = {}
    margin = full_run_margin(cfg, P, cond, n)
    np.savez_compressed(os.path.join(GOLDEN_DIR, name), meta=meta(cfg, seed, init, min_logit_margin=margin),
                        codes_top=ct.numpy(), codes_bot=cb.numpy(), **extra)
    print(name, "min greedy margin over the run", margin)


def golden_stage1(name, seed=1, B=2):
    """SURVEY.md 8f-1: pixels of the UNMODIFIED `SimRQGAN2Generator.decode_code` (generator.py:323-367) for a small HQ-VAE
    (oracle.s1_oracle.TINY_S1: every decoder stage present - mid attention, an attention level, channel-changing blocks
    with nin_shortcut, four upsample convs) on random code grids; weights are regenerated from (cfg, seed)."""
    from oracle import s1_oracle as S1
    cfg = S1.TINY_S1
    P = S1.make_params(cfg, seed=seed)
    model = R.build_reference_stage1(cfg, P)
    g = torch.Generator().manual_seed(seed + 100)
    h = cfg.latent_res // 2
    ct = torch.randint(0, cfg.n_embed, (B, h, h), generator=g)
    cb = torch.randint(0, cfg.n_embed, (B, 2 * h, 2 * h), generator=g)
    with torch.no_grad():
        px = model.decode_code(ct, cb)
    np.savez_compressed(os.path.join(GOLDEN_DIR, name),
                        meta=np.array(json.dumps(dict(config=cfg.to_dict(), seed=seed, torch=torch.__version__,
                                                      reference="SimRQGAN2Generator.decode_code, CPU fp32"))),
                        code_t=ct.numpy(), code_b=cb.numpy(), pixels=px.numpy().astype(np.float32))
    print(name, "pixels", tuple(px.shape), "mean |x|", float(px.abs().mean()))


def golden_level3(cfg, name, seed, labels, S=24):
    """SURVEY.md 8f-2: greedy code grids of the unmodified 3-level `HQTransformer` (decoding_type 'parallel-add') through the
    reference's own `sampling_hqtransformer` (scalar class) and, row by row with per-row classes, its `sampling_step`."""
    from oracle import hq3_oracle as O3
    P = O3.make_params(cfg, seed=seed)
    model = R.build_reference_hq3(cfg, P)
    g3 = dict(top_k=[1, 1, 1], top_p=[1.0, 1.0, 1.0], softmax_temperature=[1.0, 1.0, 1.0])
    labels_t = torch.tensor(labels, dtype=torch.long)
    sos = model.sos(labels_t).unsqueeze(1)
    levels, past = None, None
    for cnt in range(S):
        if levels is None:
            codes, pos = [None, None, None], None
        else:
            codes = [levels[0][:, cnt - 1:cnt], levels[1][:, cnt - 1:cnt, :], levels[2][:, cnt - 1:cnt, :]]
            pos = torch.full((len(labels), 1), cnt - 1, dtype=torch.long)
        step, present = model.sampling_step(sos=sos, codes=codes, pos_codes=pos, use_fp16=False, past=past, **g3)
        present = torch.stack(present).clone()
        past = [present] if past is None else past + [present]
        levels = step if levels is None else [torch.cat([a, b], 1) for a, b in zip(levels, step)]
    scalar = R.reference_sample_hq3(model, 2, int(labels[-1]), max_seq_len=S, **g3)
    assert all(torch.equal(s[0], l[-1]) for s, l in zip(scalar, levels))
    _, lg = O3.sample(P, cfg, labels_t, len(labels), top_k=(1, 1, 1), max_seq_len=S, return_logits=True)
    margin = min(min_margin(lg[:, :, 0, : cfg.vocab_sizes[0]]), min_margin(lg[:, :, 1:5, : cfg.vocab_sizes[1]]),
                 min_margin(lg[:, :, 5:, : cfg.vocab_sizes[2]]))
    np.savez_compressed(os.path.join(GOLDEN_DIR, name), meta=meta(cfg, seed, "rich", min_logit_margin=margin),
                        labels=np.asarray(labels, dtype=np.int64), codes_top=levels[0].numpy(), codes_mid=levels[1].numpy(),
                        codes_bot=levels[2].numpy())
    print(name, "min greedy margin over the run", margin)


def golden_filters(name):
    """Known answers of cutoff_topk_logits / cutoff_topp_probs (sampling.py:12-37) incl. ties."""
    _, S = R.import_reference()
    g = torch.Generator().manual_seed(11)
    out = {}
    logits = torch.randn(6, 512, generator=g)
    logits[1, 100] = logits[1, 7] = logits[1].max() + 1.0                   # tie at the max
    logits[2, :] = torch.round(logits[2, :] * 2) / 2                        # heavy ties everywhere
    for k in (1, 2, 5, 64, 512):
        out[f"topk_{k}"] = S.cutoff_topk_logits(logits.clone(), k).numpy()
    out["topk_in"] = logits.numpy()
    probs = torch.softmax(torch.randn(6, 512, generator=g) * 2.0, dim=-1)
    probs[0, :4] = torch.tensor([0.5, 0.3, 0.15, 0.05]) * probs[0, :4].sum() / 1.0
    small = torch.tensor([[0.5, 0.3, 0.15, 0.05], [0.25, 0.25, 0.25, 0.25], [0.97, 0.01, 0.01, 0.01]])
    for p in (0.5, 0.8, 0.95, 1.0):
        out[f"topp_{p}"] = S.cutoff_topp_probs(probs.clone(), p).numpy()
        out[f"topp_small_{p}"] = S.cutoff_topp_probs(small.clone(), p).numpy()
    out["topp_in"] = probs.numpy()
    out["topp_small_in"] = small.numpy()
    np.savez_compressed(os.path.join(GOLDEN_DIR, name), meta=np.array(json.dumps(dict(torch=torch.__version__))), **out)
    print(name, "done")


SKW = dict(top_k_top=8, top_p_top=0.9, top_k_bot=16, top_p_bot=0.95, softmax_temperature=[0.9, 1.1])
# seeded runs that tests/test_oracle_golden.py compares with these files, and with the live reference when it is present
LIVE_CHECKS = {
    "tiny_cls_scalar_class.npz": [
        dict(run="greedy", cfg={}, seed=11, cond=4, B=3, S=16, torch_seed=None, kw=GREEDY),
        dict(run="stochastic", cfg={}, seed=11, cond=2, B=3, S=8, torch_seed=5,
             kw=dict(top_k_top=20, top_p_top=0.9, top_k_bot=30, top_p_bot=0.8, softmax_temperature=[0.9, 1.2]))],
    "tiny_variants_stochastic.npz": [
        dict(run="top2bot", cfg=dict(model_type="top2bot"), seed=3, cond=4, B=3, S=6, torch_seed=5, kw=SKW),
        dict(run="bidirectional", cfg=dict(model_type="bidirectional"), seed=3, cond=4, B=3, S=6, torch_seed=5, kw=SKW),
        dict(run="reduce_2d_uncond", cfg=dict(embedding_type="reduce", position_embedding="2d", cond="uncond"), seed=3,
             cond=None, B=3, S=6, torch_seed=5, kw=SKW)],
    "tiny3_cls_stochastic.npz": [
        dict(run="stochastic", cfg={}, seed=56, cond=4, B=3, S=5, torch_seed=5,
             kw=dict(top_k=[8, 16, 32], top_p=[0.9, 0.95, 0.8], softmax_temperature=[0.9, 1.1, 1.0]))],
}


def live_check_run(name, run, reference=False):
    """Code grids of one LIVE_CHECKS run: the oracle's, or with reference=True the unmodified reference's (on CPU, the same
    weights and torch seed)."""
    if name.startswith("tiny3"):
        from oracle import hq3_oracle as O3
        cfg = O3.HQ3Config.from_dict({**O3.TINY3.to_dict(), **run["cfg"]})
        P = O3.make_params(cfg, seed=run["seed"])
    else:
        cfg = O.HQConfig(**{**O.TINY.to_dict(), **run["cfg"]})
        P = O.make_params(cfg, seed=run["seed"], init="rich")
    if run["torch_seed"] is not None:
        torch.manual_seed(run["torch_seed"])
    S = run["S"]
    if name.startswith("tiny3"):
        if reference:
            return R.reference_sample_hq3(R.build_reference_hq3(cfg, P), run["B"], run["cond"], max_seq_len=S, **run["kw"])
        return O3.sample(P, cfg, run["cond"], run["B"], max_seq_len=S, **run["kw"])
    if reference:
        return R.reference_sample(R.build_reference_model(cfg, P), run["B"], run["cond"], max_seq_len=S, **run["kw"])
    return O.sample(P, cfg, run["cond"], run["B"], max_seq_len=S, **run["kw"])


def golden_live_checks():
    """Known answers of the LIVE_CHECKS runs, so that a checkout without the reference tree still compares with them.
    The grids are the oracle's; the live tests showed them bit-identical to the unmodified reference's on exactly these
    inputs, and when the reference tree is present every run is checked against it again before anything is written."""
    checked = R.reference_available()
    for name, runs in LIVE_CHECKS.items():
        out = {}
        for run in runs:
            got = live_check_run(name, run)
            if checked:
                assert all(torch.equal(a, b) for a, b in zip(got, live_check_run(name, run, reference=True))), (name, run)
            for level, codes in zip(("top", "mid", "bot") if len(got) == 3 else ("top", "bot"), got):
                out[f"{run['run']}_{level}"] = codes.numpy()
        src = ("oracle output, checked bit-identical to the reference on these inputs when written" if checked else
               "oracle output; the live tests found the oracle bit-identical to the reference on these inputs")
        np.savez_compressed(os.path.join(GOLDEN_DIR, name),
                            meta=np.array(json.dumps(dict(torch=torch.__version__, runs=runs, source=src))), **out)
        print(name, "done", "(re-checked against the reference)" if checked else "")


def main():
    if "--live-checks" in sys.argv:
        golden_live_checks()
        return 0
    if not R.reference_available():
        print("reference tree absent - goldens can only be generated in the build container", file=sys.stderr)
        return 1
    os.makedirs(GOLDEN_DIR, exist_ok=True)
    torch.manual_seed(0)
    torch.set_num_threads(max(1, os.cpu_count() or 1))
    if "--level3" in sys.argv or "--all" in sys.argv:
        from oracle import hq3_oracle as O3
        # 24 positions x 21 codes x 3 rows = 1512 greedy decisions; seed searched (oracle) for a margin >= 2e-4 over all of them
        golden_level3(O3.TINY3, "tiny3_cls_greedy.npz", seed=56, labels=[3, 9, 0], S=24)
        if "--all" not in sys.argv:
            return 0
    if "--stage1" in sys.argv or "--all" in sys.argv:
        golden_stage1("s1_tiny_decode.npz")
        if "--all" not in sys.argv:
            return 0
    if "--variants" in sys.argv or "--all" in sys.argv:
        # seeds searched (oracle) for a greedy margin >= 2e-4 over the whole run, as for the other goldens
        V = lambda **kw: O.HQConfig(**{**O.TINY.to_dict(), **kw})
        golden_variant(V(embedding_type="reduce", cond="uncond"), "tiny_reduce_uncond_greedy.npz", seed=21, init="rich", B=2)
        golden_variant(V(position_embedding="2d"), "tiny_pos2d_cls_greedy.npz", seed=31, init="rich", labels=[1, 8, 3])
        golden_variant(V(model_type="top2bot"), "tiny_top2bot_cls_greedy.npz", seed=31, init="rich", labels=[5, 0, 9])
        golden_variant(V(model_type="bidirectional"), "tiny_bidir_cls_greedy.npz", seed=24, init="rich", labels=[2, 7, 4])
        golden_variant(O.HQConfig(**{**O.ASYM.to_dict(), "model_type": "top2bot", "embedding_type": "reduce",
                                     "position_embedding": "2d"}), "asym_top2bot_reduce_pos2d_greedy.npz", seed=62,
                       init="rich", labels=[6, 1, 4, 0])
        if "--all" not in sys.argv:
            return 0
    if "--full-size" in sys.argv or "--all" in sys.argv:       # ~1 min of CPU: the reference at ImageNet-L12 size
        golden_cls_full_size(O.IMAGENET_L12, "l12_cls_greedy_b4.npz", seed=0, labels=[166, 721, 312, 49])   # margin 1.6e-4 (label sets searched for >= 1e-4)
        if "--all" not in sys.argv:
            return 0
    golden_cls(O.SMALL, "small_cls_greedy.npz", seed=5, init="rich", labels=[0, 1, 2, 3])
    golden_cls(O.TINY, "tiny_cls_greedy.npz", seed=7, init="reference", labels=[9, 4, 4, 0, 7])
    golden_cls(O.ASYM, "asym_cls_greedy.npz", seed=4, init="rich", labels=[0, 3, 6, 2, 5])
    golden_txt(O.HQConfig(**{**O.TINY.to_dict(), "cond": "txt"}), "tiny_txt_greedy.npz", seed=2, init="rich", B=3)
    golden_txt(O.HQConfig(**{**O.ASYM.to_dict(), "cond": "txt"}), "asym_txt_greedy.npz", seed=6, init="rich", B=2)
    golden_uncond(O.HQConfig(**{**O.TINY.to_dict(), "cond": "uncond"}), "tiny_uncond_stochastic.npz", seed=3,
                  init="rich", B=4)
    golden_filters("filters.npz")
    return 0


if __name__ == "__main__":
    sys.exit(main())
