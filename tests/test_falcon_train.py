"""The Falcon-7B family (examples/falcon-7b-instruct/: the reference imports and serves it; a Model with a
trainer image fine-tunes any imported base model, internal/controller/model_controller.go) through the CUDA
fine-tune engine, against two real optimiser steps of HF FalconForCausalLM + torch.optim.AdamW with the
Trainer's decay groups (tests/golden/falcon_tiny_train.npz, oracle/make_golden.py run_falcon_train) and the
fp32 oracle (oracle/falcon_oracle.py train_step, pinned to that golden on CPU).

What this layout adds to the Llama / OPT paths: multi-query attention backward (every query head's dK / dV
lands on the one shared key/value head), the parallel block (attention and MLP read the SAME LayerNorm
output: its gradient is the sum of both branches), exact GeLU, 64-wide heads stored padded to 128 with RoPE
rotating only the first 64 columns, and a tied head on an embedding WITHOUT padding_idx.

Tolerances as tests/test_engine.py: loss / grad-norm / updated weights 1e-3, logits 1.5e-2, gradients 3e-2
relative Frobenius per tensor (bf16 compute vs fp32 golden; GeLU is smooth, no ReLU-style mask flips)."""
import numpy as np
import pytest

from oracle import falcon_oracle as FO
from util import bf16_bits, rel_err

pytestmark = pytest.mark.gpu


def _load():
    from runbooks_b200.engine import FalconArch
    fx = np.load("tests/golden/falcon_tiny_train.npz")
    V, d, L, H, dh = (int(x) for x in fx["arch"])
    oa = FO.FalconArch(vocab_size=V, hidden_size=d, num_layers=L, num_heads=H, head_dim=dh)
    arch = FalconArch(V, d, 4 * d, L, H, max_seq_len=fx["ids"].shape[1])
    return fx, oa, arch, FO.seeded_params(oa, int(fx["seed"]), std=float(fx["std"]))


def _engine(arch, params, micro_batch, **kw):
    from runbooks_b200.engine import Engine
    e = Engine(0)
    e.init_model(arch, micro_batch=micro_batch, training=True, **kw)
    e.load_state_dict(params)
    return e


def test_falcon_load_read_round_trip_through_the_padded_layout():
    fx, oa, arch, params = _load()
    e = _engine(arch, params, 2)
    assert {n for n, _ in e.params()} == set(params)
    for name, shape in e.params():
        assert tuple(shape) == params[name].shape, name
        assert np.array_equal(e.read_tensor(name, shape), params[name]), name
        assert np.array_equal(e.read_tensor(name, shape, bf16_bits=True), bf16_bits(params[name])), name
    e.close()


def test_falcon_forward_logits():
    fx, oa, arch, params = _load()
    e = _engine(arch, params, 2)
    logits, nll, _ = e.forward(fx["ids"], fx["labels"])
    err = rel_err(logits.reshape(-1)[::int(fx["logits_stride"])], fx["logits_sample"])
    print(f"falcon: logits rel_err {err:.3e}")
    assert err < 1.5e-2
    e.close()


def test_falcon_gradients_match_hf():
    fx, oa, arch, params = _load()
    e = _engine(arch, params, 2)
    loss = e.forward_backward(fx["ids"], fx["labels"])
    assert abs(loss - float(fx["loss"])) < 1e-3 * float(fx["loss"])
    ref = FO.train_step(params, fx["ids"], fx["labels"], oa)["grads"]
    rows = []
    for name, shape in e.params():
        g = e.read_state(name, shape, "grad")
        rows.append((rel_err(g, ref[name]), name))
        gn = float(np.linalg.norm(g.astype(np.float64)))
        assert abs(gn - float(fx["gradnorm/" + name])) < 1e-2 * float(fx["gradnorm/" + name]), name
    rows.sort(reverse=True)
    for err, name in rows[:4]:
        print(f"falcon grad {name:58s} rel_err {err:.3e}")
    for err, name in rows:
        assert err < 3e-2, (name, err)
    # no padding_idx (modeling_falcon.py:680): the row of config.pad_token_id gets its lookup gradient too
    tname = "transformer.word_embeddings.weight"
    g = e.read_state(tname, params[tname].shape, "grad")
    assert rel_err(g[3], fx["pad_row_grad"]) < 3e-2
    e.close()


@pytest.mark.parametrize("micro", ["full", "accumulate"])
def test_falcon_two_train_steps_match_hf(micro):
    fx, oa, arch, params = _load()
    lr1, lr2 = (float(x) for x in fx["lrs"])
    e = _engine(arch, params, 2 if micro == "full" else 1, weight_decay=float(fx["weight_decay"]))
    loss1, gn1 = e.train_step(fx["ids"], fx["labels"], lr=lr1)
    loss2, gn2 = e.train_step(fx["ids2"], fx["labels2"], lr=lr2)
    print(f"falcon/{micro}: loss {loss1:.6f}/{loss2:.6f} (HF {float(fx['loss']):.6f}/{float(fx['loss2']):.6f}) "
          f"gnorm {gn1:.5f}/{gn2:.5f} (HF {float(fx['gnorm']):.5f}/{float(fx['gnorm2']):.5f})")
    assert abs(loss1 - float(fx["loss"])) < 1e-3 * float(fx["loss"])
    assert abs(loss2 - float(fx["loss2"])) < 1e-3 * float(fx["loss2"])
    assert abs(gn1 - float(fx["gnorm"])) < 5e-3 * float(fx["gnorm"])
    assert abs(gn2 - float(fx["gnorm2"])) < 5e-3 * float(fx["gnorm2"])
    worst = 0.0
    for name, shape in e.params():
        w = e.read_state(name, shape, "master").reshape(-1)[::17]
        worst = max(worst, rel_err(w, fx["param2/" + name]))
        wb = e.read_tensor(name, shape, bf16_bits=True).reshape(-1)[::17]
        assert np.array_equal(wb, bf16_bits(w)), name
    print(f"falcon/{micro}: updated weights rel_err {worst:.3e}")
    # the golden's learning rates (1e-3 / 5e-4) exist to make the decay groups visible: an Adam step moves every
    # weight by ~lr * sign(g), so the sign noise of near-zero bf16 gradients is amplified 20x relative to the
    # reference's 5e-5 (tests/test_engine.py's trainer golden: same effect). The 1e-3 bar is checked at the
    # reference's learning rate below.
    assert worst < 1e-2
    e.close()


def test_falcon_two_train_steps_at_the_reference_learning_rate():
    """lr 5e-5 / 2.5e-5 (HF Trainer default, linear decay), weight decay 0.01, against the fp32 oracle (pinned to
    the HF golden on CPU): updated weights within 1e-3 (north_star)."""
    fx, oa, arch, params = _load()
    e = _engine(arch, params, 2, weight_decay=0.01)
    e.train_step(fx["ids"], fx["labels"], lr=5e-5)
    loss2, gn2 = e.train_step(fx["ids2"], fx["labels2"], lr=2.5e-5)
    r1 = FO.train_step(params, fx["ids"], fx["labels"], oa, lr=5e-5, step=1, weight_decay=0.01)
    r2 = FO.train_step(r1["params"], fx["ids2"], fx["labels2"], oa, lr=2.5e-5, state=r1, step=2, weight_decay=0.01)
    assert abs(loss2 - r2["loss"]) < 1e-3 * r2["loss"] and abs(gn2 - r2["gnorm"]) < 5e-3 * r2["gnorm"]
    worst = max(rel_err(e.read_state(n, s, "master"), r2["params"][n]) for n, s in e.params())
    print(f"falcon @ lr 5e-5: updated weights rel_err {worst:.3e}")
    assert worst < 1e-3
    e.close()


def test_falcon_ln_f_is_not_decayed():
    """Trainer.get_decay_parameter_names excludes nn.LayerNorm parameters by module type: `ln_f` matches none
    of the name patterns but must not decay (the golden's no_decay list). Noise-free differential check: with
    lr-scaled decay 0.5 vs 0 the decayed matrices move by lr * wd * w, ln_f.weight by nothing."""
    fx, oa, arch, params = _load()
    out = {}
    for wd in (0.0, 0.5):
        e = _engine(arch, params, 2, weight_decay=wd)
        e.train_step(fx["ids"], fx["labels"], lr=1e-3)
        out[wd] = {n: e.read_state(n, s, "master") for n, s in e.params()}
        e.close()
    for name in out[0.0]:
        diff = out[0.0][name] - out[0.5][name]
        if name in {str(x) for x in fx["no_decay"]}:
            assert not diff.any(), name
        else:
            np.testing.assert_allclose(diff, 1e-3 * 0.5 * params[name], rtol=0, atol=2e-7 + 1e-4 * np.abs(diff).max(),
                                       err_msg=name)


def test_falcon_true_7b_width_forward_through_the_training_engine():
    """The fine-tune engine's forward at the TRUE Falcon-7B layer width (71 query heads + 1 kv head of 64,
    d 4544, ffn 18176, V 65024; 2 layers) against the real FalconForCausalLM's last-position logits
    (tests/golden/falcon_7b_width.npz). The 20-token prompts are right-padded to the 128-token tile: causal
    attention leaves the first 20 positions unaffected."""
    from runbooks_b200.engine import Engine, FalconArch
    fx = np.load("tests/golden/falcon_7b_width.npz")
    V, d, L, H, dh = (int(x) for x in fx["arch"])
    oa = FO.FalconArch(vocab_size=V, hidden_size=d, num_layers=L, num_heads=H, head_dim=dh)
    params = FO.seeded_params(oa, int(fx["seed"]), std=float(fx["std"]))
    e = Engine(0)
    e.init_model(FalconArch(V, d, 4 * d, L, H, max_seq_len=128), micro_batch=3, training=False)
    e.load_state_dict(params)
    n = fx["prompts"].shape[1]
    ids = np.zeros((3, 128), dtype=np.int64)
    ids[:, :n] = fx["prompts"]
    logits, _, _ = e.forward(ids, ids)
    last = logits.reshape(3, 128, V)[:, n - 1]
    stride = int(fx["logits_stride"])
    err = np.linalg.norm(last[:, ::stride] - fx["logits_last"]) / np.linalg.norm(fx["logits_last"])
    print(f"falcon 7B-width forward (training engine): last-position logits rel_err {err:.3e}")
    assert err < 1.5e-2
    e.close()
