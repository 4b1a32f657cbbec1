"""Pins the oracle restatement (oracle/llama_oracle.py) against numbers produced by the real
HuggingFace LlamaForCausalLM + torch.optim.AdamW path (tests/golden/, made by
oracle/make_golden.py). CPU only. fp32 vs fp32, so the bar is 2e-5 relative (reassociation)."""
import numpy as np
import pytest
import torch

from oracle import llama_oracle as O

CASES = ["llama_tiny_mha", "llama_tiny_gqa"]


def rel(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-30))


def _load(case):
    fx = np.load(f"tests/golden/{case}.npz")
    v = [int(x) for x in fx["arch"]]
    eps, theta = (float(x) for x in fx["arch_f"])
    return fx, O.Arch(*v, rms_norm_eps=eps, rope_theta=theta), int(fx["batch"][1])


@pytest.mark.parametrize("case", CASES)
def test_two_steps_match_hf(case):
    fx, a, seed = _load(case)
    params = O.seeded_params(a, seed)
    r1 = O.train_step(params, fx["ids"], fx["labels"], a, lr=5e-5, step=1)
    assert abs(r1["loss"] - float(fx["loss"])) < 2e-5 * float(fx["loss"])
    assert abs(r1["gnorm"] - float(fx["gnorm"])) < 2e-5 * float(fx["gnorm"])
    assert rel(r1["logits"], fx["logits"]) < 2e-5
    for k in params:
        assert rel(r1["grads"][k].reshape(-1)[::61], fx["grad/" + k]) < 1e-4, k
    r2 = O.train_step(r1["params"], fx["ids2"], fx["labels2"], a, lr=2.5e-5,
                      state=dict(m=r1["m"], v=r1["v"]), step=2)
    assert abs(r2["loss"] - float(fx["loss2"])) < 2e-5 * float(fx["loss2"])
    assert abs(r2["gnorm"] - float(fx["gnorm2"])) < 2e-5 * float(fx["gnorm2"])
    for k in params:
        w0 = params[k].reshape(-1)[::61]
        assert rel(r2["params"][k].reshape(-1)[::61], fx["param2/" + k]) < 1e-6, k
        # the update itself (w2 - w0), which is ~1e-3 of the weights
        assert rel(r2["params"][k].reshape(-1)[::61] - w0, fx["param2/" + k] - w0) < 2e-3, k


def test_trainer_step_semantics_match_hf():
    """The Trainer step details that round 1 got wrong, pinned by the real HF objects
    (oracle/make_golden.py run_trainer_case): num_items_in_batch on the UNSHIFTED labels
    (trainer.py:2136), nn.Embedding(padding_idx=pad_token_id), weight decay on Trainer's decay group
    only (trainer.py:1280-1290). fp32 vs fp32: tight bars."""
    fx = np.load("tests/golden/llama_tiny_trainer.npz")
    v = [int(x) for x in fx["arch"]]
    eps, theta = (float(x) for x in fx["arch_f"])
    a = O.Arch(*v, rms_norm_eps=eps, rope_theta=theta, pad_token_id=int(fx["pad_token_id"]))
    params = O.seeded_params(a, int(fx["batch"][1]))
    wd = float(fx["weight_decay"])
    lr1, lr2 = (float(x) for x in fx["lrs"])
    assert O.trainer_num_items(fx["labels"]) == int(fx["num_items"])
    assert sorted(k for k in params if not O.decays(k)) == sorted(str(x) for x in fx["no_decay"])
    r1 = O.train_step(params, fx["ids"], fx["labels"], a, lr=lr1, step=1, weight_decay=wd)
    assert abs(r1["loss"] - float(fx["loss"])) < 2e-5 * float(fx["loss"])
    assert abs(r1["gnorm"] - float(fx["gnorm"])) < 2e-5 * float(fx["gnorm"])
    assert float(np.abs(r1["grads"]["model.embed_tokens.weight"][a.pad_token_id]).max()) == 0.0
    for k in params:
        assert rel(r1["grads"][k].reshape(-1)[::61], fx["grad/" + k]) < 1e-4, k
    r2 = O.train_step(r1["params"], fx["ids2"], fx["labels2"], a, lr=lr2, state=dict(m=r1["m"], v=r1["v"]), step=2,
                      weight_decay=wd)
    assert abs(r2["loss"] - float(fx["loss2"])) < 5e-5 * float(fx["loss2"])
    for k in params:
        assert rel(r2["params"][k].reshape(-1)[::61], fx["param2/" + k]) < 2e-5, k
    # the shifted-label count (what model(ids, labels) alone divides by) is a different number here
    shifted = O.train_step(params, fx["ids"], fx["labels"], a, lr=lr1)["loss"] * int(fx["num_items"]) / int(
        (fx["labels"][:, 1:] != -100).sum())
    assert abs(shifted - float(fx["loss"])) > 1e-3 * float(fx["loss"])


def test_ops_match_hf_modules():
    fx = np.load("tests/golden/llama_ops.npz")
    y = O.rmsnorm(torch.tensor(fx["rms_x"]), torch.tensor(fx["rms_w"]), 1e-5)
    assert rel(y, fx["rms_y"]) < 1e-6
    pos = fx["rope_pos"]
    cos, sin = O.rope_cos_sin(512, 128, 10000.0)
    assert rel(cos[pos], fx["rope_cos"]) < 1e-6 and rel(sin[pos], fx["rope_sin"]) < 1e-6
    qe = O.apply_rope(torch.tensor(fx["rope_q"]), cos[pos], sin[pos])
    ke = O.apply_rope(torch.tensor(fx["rope_k"]), cos[pos], sin[pos])
    assert rel(qe, fx["rope_qe"]) < 1e-6 and rel(ke, fx["rope_ke"]) < 1e-6
    o = O.causal_attention(*(torch.tensor(fx[n]) for n in ("att_q", "att_k", "att_v")))
    assert rel(o, fx["att_o"]) < 1e-5
    loss, nll = O.causal_lm_loss(torch.tensor(fx["ce_logits"]), torch.tensor(fx["ce_labels"]))
    assert abs(float(loss) - float(fx["ce_loss"])) < 1e-6 * float(fx["ce_loss"])
    assert abs(float(nll.sum()) / 40 - float(fx["ce_loss_items40"])) < 1e-6 * float(fx["ce_loss_items40"])


def test_loss_edge_cases():
    """all-ignored rows contribute nothing; the final position never has a target."""
    lg = torch.randn(2, 8, 16, generator=torch.Generator().manual_seed(0))
    lb = torch.randint(0, 16, (2, 8), generator=torch.Generator().manual_seed(1))
    lb[1] = -100
    loss, nll = O.causal_lm_loss(lg, lb)
    assert float(nll.view(2, 8)[1].abs().sum()) == 0 and float(nll.view(2, 8)[0, -1]) == 0
    ref = torch.nn.functional.cross_entropy(lg[0, :-1], lb[0, 1:])
    assert abs(float(loss) - float(ref)) < 1e-6


def test_adamw_restatement_matches_torch():
    g = torch.Generator().manual_seed(3)
    p0 = torch.randn(1000, generator=g) * 0.02
    tp = torch.nn.Parameter(p0.clone())
    opt = torch.optim.AdamW([tp], lr=5e-5, weight_decay=0.01)
    p, m, v = p0.clone(), torch.zeros(1000), torch.zeros(1000)
    for step in range(1, 5):
        gr = torch.randn(1000, generator=g) * 1e-2
        tp.grad = gr.clone()
        opt.step()
        p, m, v = O.adamw_update(p, gr, m, v, step, 5e-5, wd=0.01)
    assert rel(p - p0, tp.detach() - p0) < 1e-5


def test_linear_schedule_matches_transformers():
    from transformers import get_linear_schedule_with_warmup
    tp = torch.nn.Parameter(torch.zeros(1))
    opt = torch.optim.AdamW([tp], lr=5e-5)
    sch = get_linear_schedule_with_warmup(opt, 0, 10)
    for i in range(10):
        assert abs(opt.param_groups[0]["lr"] - O.linear_lr(i, 10)) < 1e-12
        opt.step()
        sch.step()


def test_bf16_round_matches_torch():
    x = np.random.default_rng(0).standard_normal(10000).astype(np.float32) * 3
    assert np.array_equal(O.bf16_round(x), torch.tensor(x).bfloat16().float().numpy())


def test_hf_bf16_distance():
    """How far an HF model run in bf16 sits from its own fp32 run on the golden inputs — the
    yardstick for the logits tolerance in tests/test_engine.py (documented, loose bound)."""
    fx, a, seed = _load("llama_tiny_mha")
    params = {k: torch.tensor(v) for k, v in O.seeded_params(a, seed).items()}
    ids = torch.tensor(fx["ids"])
    with torch.no_grad():
        l32 = O.forward(params, ids, a)
        l16 = O.forward({k: v.bfloat16() for k, v in params.items()}, ids, a).float()
    d = rel(l16, l32)
    print(f"bf16-vs-fp32 logits distance of the torch path itself: {d:.3e}")
    assert 1e-4 < d < 3e-2


# ---- config #1 family (facebook/opt-125m, SURVEY.md 8 a15): oracle/opt_oracle.py vs the real OPTForCausalLM ----
def _opt_fixture():
    from oracle import opt_oracle as OO
    fx = np.load("tests/golden/opt_tiny.npz")
    a = OO.OptArch(*[int(x) for x in fx["arch"]])
    return OO, fx, a, OO.seeded_params(a, int(fx["seed"]))


def test_opt_two_steps_match_hf():
    """Two optimiser steps with -100 labels: loss, grad-norm, logits, every gradient tensor and every
    updated parameter (the tied embedding/head table gets both gradient contributions)."""
    OO, fx, a, params = _opt_fixture()
    r1 = OO.train_step(params, fx["ids"], fx["labels"], a, lr=5e-5, step=1)
    assert abs(r1["loss"] - float(fx["loss"])) < 2e-5 * abs(float(fx["loss"]))
    assert abs(r1["gnorm"] - float(fx["gnorm"])) < 2e-5 * float(fx["gnorm"])
    np.testing.assert_allclose(r1["logits"], fx["logits"], rtol=0, atol=2e-5 * np.abs(fx["logits"]).max())
    for k in params:
        g = r1["grads"][k]
        # k_proj.bias has a mathematically zero gradient (softmax ignores a per-query shift of the
        # scores): both sides hold ~1e-9 rounding noise, hence the absolute floor
        assert abs(np.linalg.norm(g) - float(fx["gradnorm/" + k])) < 1e-5 * float(fx["gradnorm/" + k]) + 1e-7, k
        np.testing.assert_allclose(g.flatten()[::17], fx["grad/" + k], rtol=0, atol=1e-5 * float(fx["gradnorm/" + k]) + 1e-7, err_msg=k)
    r2 = OO.train_step(r1["params"], fx["ids2"], fx["labels2"], a, lr=2.5e-5, state=r1, step=2)
    assert abs(r2["loss"] - float(fx["loss2"])) < 2e-5 * abs(float(fx["loss2"]))
    assert abs(r2["gnorm"] - float(fx["gnorm2"])) < 2e-5 * float(fx["gnorm2"])
    for k in params:
        # k_proj.bias: its gradient is rounding noise around zero (see above) and Adam turns noise of any
        # size into steps of up to +-lr, so the reference's own value is arbitrary within the summed
        # learning rates (5e-5 + 2.5e-5). No implementation can be pinned tighter on that tensor.
        atol = 7.5e-5 if k.endswith("k_proj.bias") else 1e-6
        np.testing.assert_allclose(r2["params"][k].flatten()[::17], fx["param2/" + k], rtol=0, atol=atol, err_msg=k)


def test_opt_greedy_decode_matches_hf():
    OO, fx, a, params = _opt_fixture()
    P = {k: torch.tensor(v) for k, v in params.items()}
    with torch.no_grad():
        logits = OO.forward(P, torch.tensor(fx["prompts"]), a).numpy()
    np.testing.assert_allclose(logits, fx["gen_logits"], rtol=0, atol=2e-5 * np.abs(fx["gen_logits"]).max())
    gen = OO.greedy(params, fx["prompts"], a, fx["generated"].shape[1])
    assert (gen == fx["generated"]).all(), (gen[0].tolist(), fx["generated"][0].tolist())


def test_opt_restatement_details_matter():
    """The three things a15 calls out -- position offset 2, q scaled before the attention call, biases --
    must each change the logits by far more than the parity tolerance, so that the golden pins them."""
    OO, fx, a, params = _opt_fixture()
    P = {k: torch.tensor(v) for k, v in params.items()}
    ids = torch.tensor(fx["prompts"])
    with torch.no_grad():
        base = OO.forward(P, ids, a)
        shifted = dict(P)
        shifted["model.decoder.embed_positions.weight"] = torch.roll(P["model.decoder.embed_positions.weight"], OO.POS_OFFSET, 0)
        no_off = OO.forward(shifted, ids, a)                        # == looking positions up without the +2
        nobias = {k: (torch.zeros_like(v) if k.endswith("proj.bias") or "fc" in k and k.endswith(".bias") else v) for k, v in P.items()}
        no_b = OO.forward(nobias, ids, a)
    scale = float(base.abs().max())
    assert float((no_off - base).abs().max()) > 1e-2 * scale
    assert float((no_b - base).abs().max()) > 1e-2 * scale
    assert OO.OPT_125M.head_dim == 64 and OO.OPT_125M.max_position_embeddings + OO.POS_OFFSET == 2050
    # padding_idx: the embedding lookup gives the pad row no gradient, the tied head still does
    assert (fx["ids"] == a.pad_token_id).any(), "the fixture must contain the pad id as an ordinary input token"
    plain = OO.OptArch(a.vocab_size, a.hidden_size, a.ffn_dim, a.num_layers, a.num_heads, a.max_position_embeddings, pad_token_id=-1)
    g_pad = OO.train_step(params, fx["ids"], fx["labels"], a)["grads"]["model.decoder.embed_tokens.weight"]
    g_plain = OO.train_step(params, fx["ids"], fx["labels"], plain)["grads"]["model.decoder.embed_tokens.weight"]
    assert np.abs(g_pad - g_plain).max() > 1e-4 * np.abs(g_pad).max()


def test_falcon_two_train_steps_match_hf():
    """oracle/falcon_oracle.py train_step against two real optimiser steps of FalconForCausalLM + AdamW with the
    Trainer's decay groups (weight decay 0.5 so that a wrong group shows: `ln_f` is excluded by module type,
    not by name)."""
    from oracle import falcon_oracle as FO
    fx = np.load("tests/golden/falcon_tiny_train.npz")
    V, d, L, H, dh = (int(x) for x in fx["arch"])
    a = FO.FalconArch(vocab_size=V, hidden_size=d, num_layers=L, num_heads=H, head_dim=dh)
    params = FO.seeded_params(a, int(fx["seed"]), std=float(fx["std"]))
    assert sorted(k for k in params if not FO.decays(k)) == sorted(str(x) for x in fx["no_decay"])
    lr1, lr2 = (float(x) for x in fx["lrs"])
    wd = float(fx["weight_decay"])
    r1 = FO.train_step(params, fx["ids"], fx["labels"], a, lr=lr1, step=1, weight_decay=wd)
    assert abs(r1["loss"] - float(fx["loss"])) < 2e-5 * abs(float(fx["loss"]))
    assert abs(r1["gnorm"] - float(fx["gnorm"])) < 2e-5 * float(fx["gnorm"])
    np.testing.assert_allclose(r1["logits"].reshape(-1)[::int(fx["logits_stride"])], fx["logits_sample"], rtol=0,
                               atol=2e-5 * np.abs(fx["logits_sample"]).max())
    for k in params:
        g = r1["grads"][k]
        assert abs(np.linalg.norm(g) - float(fx["gradnorm/" + k])) < 1e-5 * float(fx["gradnorm/" + k]), k
        np.testing.assert_allclose(g.flatten()[::17], fx["grad/" + k], rtol=0, atol=1e-5 * float(fx["gradnorm/" + k]), err_msg=k)
    np.testing.assert_allclose(r1["grads"]["transformer.word_embeddings.weight"][3], fx["pad_row_grad"], rtol=0,
                               atol=1e-5 * np.abs(fx["pad_row_grad"]).max())
    assert np.abs(fx["pad_row_grad"]).max() > 0
    r2 = FO.train_step(r1["params"], fx["ids2"], fx["labels2"], a, lr=lr2, state=r1, step=2, weight_decay=wd)
    assert abs(r2["loss"] - float(fx["loss2"])) < 2e-5 * abs(float(fx["loss2"]))
    assert abs(r2["gnorm"] - float(fx["gnorm2"])) < 2e-5 * float(fx["gnorm2"])
    for k in params:
        np.testing.assert_allclose(r2["params"][k].flatten()[::17], fx["param2/" + k], rtol=0, atol=2e-5, err_msg=k)
