"""Generates tests/golden/*.npz by running the REAL HuggingFace/PyTorch path — the libraries the
reference's trainer image wraps — on seeded tiny inputs. Run here (CPU):

    python oracle/make_golden.py

The fixtures pin oracle/llama_oracle.py (tests/test_oracle_golden.py) and are what the CUDA
parity tests are ultimately anchored to. transformers.Trainer itself cannot be imported in this
image (needs `accelerate`), so the Trainer step is written out with the same torch objects
Trainer uses: model(...).loss.backward(); clip_grad_norm_(params, 1.0); AdamW(lr=5e-5,
betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0).step()  (TrainingArguments defaults).
"""
from __future__ import annotations

import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle.llama_oracle import Arch, seeded_params  # noqa: E402

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")

CASES = {
    # name: (arch, batch, seed)
    "llama_tiny_mha": (Arch(256, 256, 384, 2, 2, 2, 128, 128, 1e-5, 10000.0), 2, 11),
    "llama_tiny_gqa": (Arch(320, 512, 256, 1, 4, 2, 128, 256, 1e-6, 10000.0), 1, 12),
}
SAMPLE_STRIDE = 61  # strided samples of big tensors keep the fixtures small


def make_batch(a: Arch, B: int, seed: int):
    rng = np.random.default_rng(seed + 1000)
    ids = rng.integers(0, a.vocab_size, size=(B, a.max_seq_len), dtype=np.int64)
    labels = ids.copy()
    # mask a prompt-like prefix and a few scattered tokens with the HF ignore index
    labels[:, : a.max_seq_len // 8] = -100
    labels[rng.random(labels.shape) < 0.05] = -100
    return ids, labels


def hf_model(a: Arch, params, pad_token_id=None):
    from transformers import LlamaConfig, LlamaForCausalLM

    cfg = LlamaConfig(
        vocab_size=a.vocab_size, hidden_size=a.hidden_size, intermediate_size=a.intermediate_size,
        num_hidden_layers=a.num_layers, num_attention_heads=a.num_heads,
        num_key_value_heads=a.num_kv_heads, head_dim=a.head_dim,
        max_position_embeddings=a.max_seq_len, rms_norm_eps=a.rms_norm_eps,
        rope_parameters={"rope_type": "default", "rope_theta": a.rope_theta},
        tie_word_embeddings=False, attention_bias=False, mlp_bias=False, attention_dropout=0.0,
        pad_token_id=pad_token_id,
    )
    cfg._attn_implementation = "sdpa"
    model = LlamaForCausalLM(cfg).float()
    sd = {k: torch.tensor(v) for k, v in params.items()}
    missing, unexpected = model.load_state_dict(sd, strict=False)
    assert not unexpected and all("rotary" in m or "inv_freq" in m for m in missing), (missing, unexpected)
    return model


def run_case(name, a: Arch, B: int, seed: int):
    torch.manual_seed(0)
    torch.set_num_threads(8)
    params = seeded_params(a, seed)
    ids, labels = make_batch(a, B, seed)
    model = hf_model(a, params)
    model.train()
    out = model(input_ids=torch.tensor(ids), labels=torch.tensor(labels))
    loss = out.loss
    loss.backward()
    named = dict(model.named_parameters())
    grads = {k: p.grad.detach().clone() for k, p in named.items()}
    gnorm = float(torch.nn.utils.clip_grad_norm_(list(named.values()), 1.0))
    opt = torch.optim.AdamW(list(named.values()), lr=5e-5, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0)
    opt.step()
    # second step with a fresh batch, to exercise non-zero Adam moments and bias correction
    opt.zero_grad(set_to_none=True)
    ids2, labels2 = make_batch(a, B, seed + 7)
    out2 = model(input_ids=torch.tensor(ids2), labels=torch.tensor(labels2))
    out2.loss.backward()
    gnorm2 = float(torch.nn.utils.clip_grad_norm_(list(named.values()), 1.0))
    for g in opt.param_groups:
        g["lr"] = 2.5e-5
    opt.step()

    fx = dict(
        arch=np.array([a.vocab_size, a.hidden_size, a.intermediate_size, a.num_layers, a.num_heads,
                       a.num_kv_heads, a.head_dim, a.max_seq_len], dtype=np.int64),
        arch_f=np.array([a.rms_norm_eps, a.rope_theta], dtype=np.float64),
        batch=np.array([B, seed], dtype=np.int64),
        ids=ids, labels=labels, ids2=ids2, labels2=labels2,
        loss=np.float32(loss.item()), gnorm=np.float32(gnorm),
        loss2=np.float32(out2.loss.item()), gnorm2=np.float32(gnorm2),
        logits=out.logits.detach().numpy().astype(np.float32),
    )
    for k in named:
        fx["gradnorm/" + k] = np.float32(grads[k].norm().item())
        fx["grad/" + k] = grads[k].flatten()[::SAMPLE_STRIDE].numpy().copy()
        fx["param2/" + k] = named[k].detach().flatten()[::SAMPLE_STRIDE].numpy().copy()
    os.makedirs(OUT, exist_ok=True)
    path = os.path.join(OUT, name + ".npz")
    np.savez_compressed(path, **fx)
    print(f"{name}: loss {loss.item():.6f} gnorm {gnorm:.6f} loss2 {out2.loss.item():.6f} -> {path} "
          f"({os.path.getsize(path) / 1024:.0f} KiB)")


def run_trainer_case():
    """The three places where round 1 deviated from the Trainer step, pinned by the real HF objects:
    (1) num_items_in_batch counted on the UNSHIFTED labels (trainer.py:2136) and passed to the model,
    (2) config.pad_token_id -> nn.Embedding(padding_idx) (the pad row gets no lookup gradient),
    (3) weight_decay = 0.01 with Trainer's decay / no-decay groups (trainer.py:1280-1290,
        trainer_pt_utils.get_parameter_names)."""
    from transformers.trainer_pt_utils import get_parameter_names

    a = Arch(256, 256, 384, 2, 2, 2, 128, 128, 1e-5, 10000.0, pad_token_id=3)
    B, seed, wd = 2, 41, 0.5   # lr 1e-3 x wd 0.5: the decay is 5e-4 per step, well above the bf16 noise floor
    torch.manual_seed(0)
    torch.set_num_threads(8)
    params = seeded_params(a, seed)
    rng = np.random.default_rng(seed + 1000)

    def batch():
        ids = rng.integers(0, a.vocab_size, size=(B, a.max_seq_len), dtype=np.int64)
        ids[:, 5] = a.pad_token_id
        ids[0, 77] = a.pad_token_id
        labels = ids.copy()                    # packed plain text: every label counts, incl. position 0
        labels[1, 30:41] = -100
        return ids, labels

    model = hf_model(a, params, pad_token_id=a.pad_token_id)
    assert model.model.embed_tokens.padding_idx == a.pad_token_id
    model.train()
    named = dict(model.named_parameters())
    forbidden = [r"bias", r"layernorm", r"rmsnorm", r"(?:^|\.)norm(?:$|\.)", r"_norm(?:$|\.)"]
    decay_names = set(get_parameter_names(model, [torch.nn.LayerNorm], forbidden))
    opt = torch.optim.AdamW([
        {"params": [p for n, p in named.items() if n in decay_names], "weight_decay": wd},
        {"params": [p for n, p in named.items() if n not in decay_names], "weight_decay": 0.0},
    ], lr=1e-3, betas=(0.9, 0.999), eps=1e-8)
    fx = dict(arch=np.array([a.vocab_size, a.hidden_size, a.intermediate_size, a.num_layers, a.num_heads,
                             a.num_kv_heads, a.head_dim, a.max_seq_len], dtype=np.int64), lrs=np.array([1e-3, 5e-4]),
              arch_f=np.array([a.rms_norm_eps, a.rope_theta], dtype=np.float64),
              batch=np.array([B, seed], dtype=np.int64), pad_token_id=np.int64(a.pad_token_id),
              weight_decay=np.float64(wd), no_decay=np.array(sorted(set(named) - decay_names)))
    for step, lr in ((1, 1e-3), (2, 5e-4)):
        ids, labels = batch()
        n = torch.tensor(int((labels != -100).sum()))
        out = model(input_ids=torch.tensor(ids), labels=torch.tensor(labels), num_items_in_batch=n)
        out.loss.backward()
        if step == 1:
            grads = {k: p.grad.detach().clone() for k, p in named.items()}
            fx["logits"] = out.logits.detach().numpy().astype(np.float32)
        gnorm = float(torch.nn.utils.clip_grad_norm_(list(named.values()), 1.0))
        for g in opt.param_groups:
            g["lr"] = lr
        opt.step()
        opt.zero_grad(set_to_none=True)
        sfx = "" if step == 1 else "2"
        fx["ids" + sfx], fx["labels" + sfx] = ids, labels
        fx["loss" + sfx], fx["gnorm" + sfx] = np.float32(out.loss.item()), np.float32(gnorm)
        fx["num_items" + sfx] = np.int64(int(n))
    for k in named:
        fx["gradnorm/" + k] = np.float32(grads[k].norm().item())
        fx["grad/" + k] = grads[k].flatten()[::SAMPLE_STRIDE].numpy().copy()
        fx["param2/" + k] = named[k].detach().flatten()[::SAMPLE_STRIDE].numpy().copy()
    fx["pad_row_grad"] = grads["model.embed_tokens.weight"][a.pad_token_id].numpy().copy()
    path = os.path.join(OUT, "llama_tiny_trainer.npz")
    np.savez_compressed(path, **fx)
    print(f"llama_tiny_trainer: loss {float(fx['loss']):.6f} gnorm {float(fx['gnorm']):.6f} num_items {int(fx['num_items'])} "
          f"no_decay {len(fx['no_decay'])} tensors -> {path} ({os.path.getsize(path) / 1024:.0f} KiB)")


def run_falcon_7b_width():
    """Config #4 at the TRUE Falcon-7B layer width (d 4544, 71 query heads + 1 kv head of 64, ffn 18176,
    V 65024), 2 layers: the shapes the toy golden cannot reach -- 71 is not a multiple of the decode
    attention's 8-head group, 4544 is not a multiple of 128, split-K runs at K = 18176. Prompt logits
    (strided sample), greedy continuation and the fp32 top-2 margin of every generated step, from the
    real FalconForCausalLM. Parameters are re-created from the seed by the test (710 M values)."""
    from transformers import FalconConfig, FalconForCausalLM
    from oracle import falcon_oracle as FO

    a = FO.FalconArch(vocab_size=65024, hidden_size=4544, num_layers=2, num_heads=71, head_dim=64)
    # one layer's std 0.12 random matrices at this width would saturate everything: scale as 1/sqrt(fan_in)
    params = FO.seeded_params(a, 23, std=0.015)
    cfg = FalconConfig(vocab_size=a.vocab_size, hidden_size=a.hidden_size, num_hidden_layers=a.num_layers,
                       num_attention_heads=a.num_heads, multi_query=True, parallel_attn=True, bias=False,
                       new_decoder_architecture=False, alibi=False, layer_norm_epsilon=1e-5,
                       max_position_embeddings=2048, tie_word_embeddings=True, hidden_dropout=0.0,
                       attention_dropout=0.0)
    cfg._attn_implementation = "sdpa"
    torch.set_num_threads(8)
    model = FalconForCausalLM(cfg).float().eval()
    sd = {k: torch.tensor(v) for k, v in params.items()}
    sd["lm_head.weight"] = sd["transformer.word_embeddings.weight"]
    missing, unexpected = model.load_state_dict(sd, strict=False)
    assert not unexpected and all("rotary" in m or "inv_freq" in m for m in missing), (missing, unexpected)
    rng = np.random.default_rng(78)
    prompts = rng.integers(0, a.vocab_size, size=(3, 20), dtype=np.int64)
    n_new = 8
    with torch.no_grad():
        logits = model(torch.tensor(prompts)).logits.numpy()
        ids = torch.tensor(prompts)
        gen, margins = [], []
        for _ in range(n_new):
            lg = model(ids).logits[:, -1]
            top2 = torch.topk(lg, 2, dim=-1).values
            margins.append((top2[:, 0] - top2[:, 1]).numpy())
            nxt = lg.argmax(-1, keepdim=True)
            gen.append(nxt.numpy())
            ids = torch.cat([ids, nxt], dim=1)
    gen = np.concatenate(gen, axis=1)
    path = os.path.join(OUT, "falcon_7b_width.npz")
    np.savez_compressed(path, arch=np.array([a.vocab_size, a.hidden_size, a.num_layers, a.num_heads, a.head_dim]),
                        seed=np.int64(23), std=np.float64(0.015), prompts=prompts,
                        logits_last=logits[:, -1, ::8].astype(np.float32), logits_stride=np.int64(8),
                        logits_last_absmax=np.abs(logits[:, -1]).max(-1).astype(np.float32),
                        logits_norm=np.linalg.norm(logits[:, -1].astype(np.float64), axis=-1),
                        generated=gen, margins=np.stack(margins, 1).astype(np.float32))
    print(f"falcon_7b_width -> {path} ({os.path.getsize(path) / 1024:.0f} KiB); generated[0] = {gen[0].tolist()} "
          f"margins[0] = {np.stack(margins, 1)[0].round(3).tolist()}")


def run_ops():
    """Per-op fixtures from the HF modules themselves."""
    from transformers.loss.loss_utils import ForCausalLMLoss
    from transformers.models.llama.modeling_llama import (LlamaRMSNorm, LlamaRotaryEmbedding,
                                                          apply_rotary_pos_emb)
    from transformers import LlamaConfig

    rng = np.random.default_rng(5)
    fx = {}
    x = rng.standard_normal((6, 256)).astype(np.float32)
    w = (1 + 0.1 * rng.standard_normal(256)).astype(np.float32)
    n = LlamaRMSNorm(256, eps=1e-5)
    n.weight.data = torch.tensor(w)
    fx["rms_x"], fx["rms_w"] = x, w
    fx["rms_y"] = n(torch.tensor(x)).detach().numpy()

    cfg = LlamaConfig(hidden_size=256, num_attention_heads=2, head_dim=128,
                      max_position_embeddings=512,
                      rope_parameters={"rope_type": "default", "rope_theta": 10000.0})
    rot = LlamaRotaryEmbedding(cfg)
    q = rng.standard_normal((1, 2, 512, 128)).astype(np.float32)
    k = rng.standard_normal((1, 2, 512, 128)).astype(np.float32)
    pos = torch.arange(512)[None]
    cos, sin = rot(torch.tensor(q), pos)
    qe, ke = apply_rotary_pos_emb(torch.tensor(q), torch.tensor(k), cos, sin)
    sel = np.array([0, 1, 2, 3, 64, 127, 128, 255, 300, 511])  # positions kept in the fixture
    fx["rope_pos"] = sel
    fx["rope_q"], fx["rope_k"] = q[:, :, sel], k[:, :, sel]
    fx["rope_qe"], fx["rope_ke"] = qe.numpy()[:, :, sel], ke.numpy()[:, :, sel]
    fx["rope_cos"], fx["rope_sin"] = cos[0].numpy()[sel], sin[0].numpy()[sel]

    qa = rng.standard_normal((1, 2, 128, 128)).astype(np.float32)
    ka = rng.standard_normal((1, 1, 128, 128)).astype(np.float32)
    va = rng.standard_normal((1, 1, 128, 128)).astype(np.float32)
    o = torch.nn.functional.scaled_dot_product_attention(
        torch.tensor(qa), torch.tensor(ka).repeat_interleave(2, 1), torch.tensor(va).repeat_interleave(2, 1),
        is_causal=True, scale=128 ** -0.5)
    fx["att_q"], fx["att_k"], fx["att_v"], fx["att_o"] = qa, ka, va, o.numpy()

    lg = (3 * rng.standard_normal((2, 16, 64))).astype(np.float32)
    lb = rng.integers(0, 64, size=(2, 16), dtype=np.int64)
    lb[0, :3] = -100
    lb[1, 7] = -100
    loss = ForCausalLMLoss(torch.tensor(lg), torch.tensor(lb), vocab_size=64)
    loss_n = ForCausalLMLoss(torch.tensor(lg), torch.tensor(lb), vocab_size=64,
                             num_items_in_batch=torch.tensor(40))
    fx["ce_logits"], fx["ce_labels"] = lg, lb
    fx["ce_loss"], fx["ce_loss_items40"] = np.float32(loss.item()), np.float32(loss_n.item())
    path = os.path.join(OUT, "llama_ops.npz")
    np.savez_compressed(path, **fx)
    print(f"ops -> {path} ({os.path.getsize(path) / 1024:.0f} KiB)")


def run_falcon():
    """Tiny falcon-7b-layout model: prompt logits + greedy generation from the real HF classes."""
    from transformers import FalconConfig, FalconForCausalLM
    from oracle import falcon_oracle as FO

    a = FO.FalconArch(vocab_size=512, hidden_size=256, num_layers=2, num_heads=4, head_dim=64)
    params = FO.seeded_params(a, 21)
    cfg = FalconConfig(vocab_size=a.vocab_size, hidden_size=a.hidden_size, num_hidden_layers=a.num_layers,
                       num_attention_heads=a.num_heads, multi_query=True, parallel_attn=True, bias=False,
                       new_decoder_architecture=False, alibi=False, layer_norm_epsilon=1e-5,
                       max_position_embeddings=256, tie_word_embeddings=True, hidden_dropout=0.0,
                       attention_dropout=0.0)
    cfg._attn_implementation = "sdpa"
    model = FalconForCausalLM(cfg).float().eval()
    sd = {k: torch.tensor(v) for k, v in params.items()}
    sd["lm_head.weight"] = sd["transformer.word_embeddings.weight"]
    missing, unexpected = model.load_state_dict(sd, strict=False)
    assert not unexpected and all("rotary" in m or "inv_freq" in m for m in missing), (missing, unexpected)
    rng = np.random.default_rng(77)
    prompts = rng.integers(0, a.vocab_size, size=(3, 24), dtype=np.int64)
    with torch.no_grad():
        logits = model(torch.tensor(prompts)).logits.numpy()
        gen = model.generate(torch.tensor(prompts), max_new_tokens=12, do_sample=False,
                             pad_token_id=0).numpy()[:, prompts.shape[1]:]
    path = os.path.join(OUT, "falcon_tiny.npz")
    np.savez_compressed(path, arch=np.array([a.vocab_size, a.hidden_size, a.num_layers, a.num_heads, a.head_dim]),
                        seed=np.int64(21), prompts=prompts, logits=logits.astype(np.float32), generated=gen)
    print(f"falcon -> {path} ({os.path.getsize(path) / 1024:.0f} KiB); generated[0] = {gen[0].tolist()}")


def run_opt():
    """Tiny opt-125m-family model (SURVEY.md 8 a15) through the real OPTForCausalLM: two optimiser
    steps with -100 labels (logits, gradients, updated weights) and a greedy continuation."""
    from transformers import OPTConfig, OPTForCausalLM
    from oracle import opt_oracle as OO

    a = OO.OptArch(vocab_size=192, hidden_size=128, ffn_dim=256, num_layers=2, num_heads=2, max_position_embeddings=128)
    params = OO.seeded_params(a, 31)
    cfg = OPTConfig(vocab_size=a.vocab_size, hidden_size=a.hidden_size, ffn_dim=a.ffn_dim, num_hidden_layers=a.num_layers,
                    num_attention_heads=a.num_heads, max_position_embeddings=a.max_position_embeddings,
                    word_embed_proj_dim=a.hidden_size, do_layer_norm_before=True, activation_function="relu",
                    enable_bias=True, dropout=0.0, attention_dropout=0.0, layerdrop=0.0, tie_word_embeddings=True)
    cfg._attn_implementation = "sdpa"
    torch.manual_seed(0)
    model = OPTForCausalLM(cfg).float()
    sd = {k: torch.tensor(v) for k, v in params.items()}
    sd["lm_head.weight"] = sd["model.decoder.embed_tokens.weight"]
    missing, unexpected = model.load_state_dict(sd, strict=False)
    assert not unexpected and not missing, (missing, unexpected)
    assert model.lm_head.weight.data_ptr() == model.model.decoder.embed_tokens.weight.data_ptr(), "head must be tied"
    rng = np.random.default_rng(32)
    B, S = 2, 128   # the CUDA attention kernels take sequence lengths that are multiples of 128

    def batch():
        ids = rng.integers(0, a.vocab_size, size=(B, S)).astype(np.int64)
        ids[0, 40] = ids[1, 7] = a.pad_token_id      # the pad row must get no lookup gradient
        labels = ids.copy()
        labels[0, :9] = -100
        labels[1, 20:27] = -100                      # row 1 keeps its FIRST label: Trainer counts it
        return ids, labels

    def n_items(lab):
        """HF Trainer's num_items_in_batch (trainer.py:2136): non-ignored UNSHIFTED labels."""
        return torch.tensor(int((lab != -100).sum()))

    ids, labels = batch()
    model.train()
    out = model(input_ids=torch.tensor(ids), labels=torch.tensor(labels), num_items_in_batch=n_items(labels))
    out.loss.backward()
    named = dict(model.named_parameters())          # tied weight appears once
    grads = {k: p.grad.detach().clone() for k, p in named.items()}
    gnorm = float(torch.nn.utils.clip_grad_norm_(list(named.values()), 1.0))
    opt = torch.optim.AdamW(list(named.values()), lr=5e-5, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0)
    opt.step()
    opt.zero_grad(set_to_none=True)
    ids2, labels2 = batch()
    out2 = model(input_ids=torch.tensor(ids2), labels=torch.tensor(labels2), num_items_in_batch=n_items(labels2))
    out2.loss.backward()
    gnorm2 = float(torch.nn.utils.clip_grad_norm_(list(named.values()), 1.0))
    for g in opt.param_groups:
        g["lr"] = 2.5e-5
    opt.step()
    fx = dict(arch=np.array([a.vocab_size, a.hidden_size, a.ffn_dim, a.num_layers, a.num_heads, a.max_position_embeddings]),
              seed=np.int64(31), ids=ids, labels=labels, ids2=ids2, labels2=labels2,
              loss=np.float32(out.loss.item()), gnorm=np.float32(gnorm), loss2=np.float32(out2.loss.item()),
              gnorm2=np.float32(gnorm2), logits=out.logits.detach().numpy().astype(np.float32))
    for k in named:
        fx["gradnorm/" + k] = np.float32(grads[k].norm().item())
        fx["grad/" + k] = grads[k].flatten()[::17].numpy().copy()
        fx["param2/" + k] = named[k].detach().flatten()[::17].numpy().copy()
    # greedy continuation from the ORIGINAL weights
    model2 = OPTForCausalLM(cfg).float().eval()
    model2.load_state_dict(sd, strict=False)
    prompts = rng.integers(0, a.vocab_size, size=(3, 16)).astype(np.int64)
    with torch.no_grad():
        gen = model2.generate(torch.tensor(prompts), max_new_tokens=10, do_sample=False, pad_token_id=1).numpy()[:, 16:]
        fx["gen_logits"] = model2(torch.tensor(prompts)).logits.numpy().astype(np.float32)
    fx["prompts"], fx["generated"] = prompts, gen
    path = os.path.join(OUT, "opt_tiny.npz")
    np.savez_compressed(path, **fx)
    print(f"opt -> {path} ({os.path.getsize(path) / 1024:.0f} KiB): loss {out.loss.item():.6f} gnorm {gnorm:.6f} "
          f"loss2 {out2.loss.item():.6f}; generated[0] = {gen[0].tolist()}")


def run_falcon_train():
    """Tiny falcon-7b-layout model through two real optimiser steps (FalconForCausalLM + torch AdamW with the
    Trainer's decay groups): multi-query attention backward (4 query heads share one key/value head), the
    parallel block's shared LayerNorm gradient, exact GeLU, the tied head."""
    from transformers import FalconConfig, FalconForCausalLM
    from transformers.trainer_pt_utils import get_parameter_names
    from oracle import falcon_oracle as FO

    a = FO.FalconArch(vocab_size=512, hidden_size=256, num_layers=2, num_heads=4, head_dim=64)
    params = FO.seeded_params(a, 41, std=0.06)
    cfg = FalconConfig(vocab_size=a.vocab_size, hidden_size=a.hidden_size, num_hidden_layers=a.num_layers,
                       num_attention_heads=a.num_heads, multi_query=True, parallel_attn=True, bias=False,
                       new_decoder_architecture=False, alibi=False, layer_norm_epsilon=1e-5,
                       max_position_embeddings=256, tie_word_embeddings=True, hidden_dropout=0.0,
                       attention_dropout=0.0, pad_token_id=3)
    cfg._attn_implementation = "sdpa"
    torch.manual_seed(0)
    model = FalconForCausalLM(cfg).float()
    sd = {k: torch.tensor(v) for k, v in params.items()}
    sd["lm_head.weight"] = sd["transformer.word_embeddings.weight"]
    missing, unexpected = model.load_state_dict(sd, strict=False)
    assert not unexpected and all("rotary" in m or "inv_freq" in m for m in missing), (missing, unexpected)
    assert model.lm_head.weight.data_ptr() == model.transformer.word_embeddings.weight.data_ptr(), "head must be tied"
    rng = np.random.default_rng(42)
    B, S, WD = 2, 128, 0.5

    def batch():
        ids = rng.integers(0, a.vocab_size, size=(B, S)).astype(np.int64)
        ids[0, 33] = ids[1, 5] = 3                   # config.pad_token_id: Falcon's embedding has no padding_idx
        labels = ids.copy()
        labels[0, :11] = -100
        labels[1, 50:61] = -100
        return ids, labels

    def n_items(lab):
        return torch.tensor(int((lab != -100).sum()))

    named = dict(model.named_parameters())
    # Trainer.get_decay_parameter_names (trainer.py:1280-1290)
    decay = [n for n in get_parameter_names(model, [torch.nn.LayerNorm], ["bias", "layernorm", "rmsnorm", "norm"])]
    groups = [{"params": [p for n, p in named.items() if n in decay], "weight_decay": WD},
              {"params": [p for n, p in named.items() if n not in decay], "weight_decay": 0.0}]
    opt = torch.optim.AdamW(groups, lr=1e-3, betas=(0.9, 0.999), eps=1e-8)
    ids, labels = batch()
    model.train()
    out = model(input_ids=torch.tensor(ids), labels=torch.tensor(labels), num_items_in_batch=n_items(labels))
    out.loss.backward()
    grads = {k: p.grad.detach().clone() for k, p in named.items()}
    gnorm = float(torch.nn.utils.clip_grad_norm_(list(named.values()), 1.0))
    opt.step()
    opt.zero_grad(set_to_none=True)
    ids2, labels2 = batch()
    out2 = model(input_ids=torch.tensor(ids2), labels=torch.tensor(labels2), num_items_in_batch=n_items(labels2))
    out2.loss.backward()
    gnorm2 = float(torch.nn.utils.clip_grad_norm_(list(named.values()), 1.0))
    for g in opt.param_groups:
        g["lr"] = 5e-4
    opt.step()
    fx = dict(arch=np.array([a.vocab_size, a.hidden_size, a.num_layers, a.num_heads, a.head_dim]), seed=np.int64(41),
              std=np.float64(0.06), weight_decay=np.float64(WD), lrs=np.array([1e-3, 5e-4]),
              ids=ids, labels=labels, ids2=ids2, labels2=labels2, loss=np.float32(out.loss.item()),
              gnorm=np.float32(gnorm), loss2=np.float32(out2.loss.item()), gnorm2=np.float32(gnorm2),
              # every 3rd logit of the flattened [B, S, V]: 3 is coprime to V, so every position and every
              # vocabulary column is still sampled, and the fixture stays under 1 MB
              logits_stride=np.int64(3),
              logits_sample=out.logits.detach().numpy().astype(np.float32).reshape(-1)[::3].copy(),
              no_decay=np.array(sorted(n for n in named if n not in decay)))
    for k in named:
        fx["gradnorm/" + k] = np.float32(grads[k].norm().item())
        fx["grad/" + k] = grads[k].flatten()[::17].numpy().copy()
        fx["param2/" + k] = named[k].detach().flatten()[::17].numpy().copy()
    fx["pad_row_grad"] = grads["transformer.word_embeddings.weight"][3].numpy().copy()
    path = os.path.join(OUT, "falcon_tiny_train.npz")
    np.savez_compressed(path, **fx)
    print(f"falcon_tiny_train -> {path} ({os.path.getsize(path) / 1024:.0f} KiB): loss {out.loss.item():.6f} "
          f"gnorm {gnorm:.6f} loss2 {out2.loss.item():.6f} gnorm2 {gnorm2:.6f}; no_decay {len(fx['no_decay'])}")


if __name__ == "__main__":
    if "--falcon-train-only" in sys.argv:
        run_falcon_train()
        sys.exit(0)
    if "--opt-only" in sys.argv:
        run_opt()
        sys.exit(0)
    if "--round2" in sys.argv:     # the fixtures added in round 2 (the others are unchanged)
        run_opt()
        run_trainer_case()
        run_falcon_7b_width()
        run_falcon_train()
        sys.exit(0)
    run_ops()
    run_falcon()
    run_opt()
    run_trainer_case()
    run_falcon_7b_width()
    run_falcon_train()
    for name, (a, B, seed) in CASES.items():
        run_case(name, a, B, seed)
