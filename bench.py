#!/usr/bin/env python
"""bench.py — tokens/sec of the Llama-2-7B fine-tune step (BASELINE.json metric) on N B200s.

    python bench.py --gpus 1 --steps 5 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference ...     # the HF/PyTorch CPU path of the reference's image

A "step" is one optimiser step of the fine-tune hot path: forward, loss, backward, (gradient
all-reduce), global-norm clip, AdamW over `per_device_batch` packed 4096-token sequences per
GPU (HF TrainingArguments default per_device_train_batch_size = 8, run as 8 accumulation
micro-steps of one sequence), synthetic token ids, random-init weights of the named arch.

Printed line (rank 0): the contract keys + `roofline` (tcgen05 GEMM kernel, CUDA-event timed
live inside the timed region) + `cpu_baseline` (the oracle port timed on host cores, N=1 only)
+ `e2e` (same metric through the public host-buffer API) + `clocks`.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "tokens/sec Llama-2-7B fine-tune at 1/2/4/8 B200; % tensor-core roofline"
FLOPS_PER_TOKEN = 42.864e9  # SURVEY.md §8d: 6*N_mm + 6*L*S*d at S=4096, no recompute credit


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(burst=d["bf16_tflops"], sustained=d["bf16_tflops_sustained"], hbm=d["hbm_gbs"],
                    source="measured")
    return dict(burst=1590.0, sustained=1400.0, hbm=6650.0, source="fallback")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                 "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
        sm, mx, reasons = [], 0.0, set()
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx = max(mx, float(r[2]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown",
                                    "sw_power_cap"), r[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except (ValueError, IndexError):
                pass
        sm.sort()
        return dict(sm_mhz=sm[len(sm) // 2] if sm else None, sm_max_mhz=mx or None,
                    reasons=sorted(reasons), samples=len(sm))


# --------------------------------------------------------------------------------------------
# CPU legs: the oracle port of the reference's HF/PyTorch path, on a bounded sample.
# ONE sample definition for both legs (`cpu_baseline` of the CUDA arm and `--impl reference`):
#   one decoder layer of true Llama-2-7B width on a FULL 4096-token sequence -- forward, backward of
#   the real loss (final norm + lm_head + cross-entropy on that layer's output), AdamW on the layer --
#   with the layer part and the head part timed separately; the step time of the 32-layer model is
#   32 x layer + head (no extrapolation in tokens: attention is quadratic in them), x 8 sequences.
# Thread count: chosen once by a short matmul sweep (a shared 128-thread host is slower AND 16x noisier
# with every thread in use than with 16-32: round 1's five runs spread 0.44 ... 7.0 tok/s).
# Reported: the MEDIAN of >= 3 repeats and their max/min spread.
# --------------------------------------------------------------------------------------------
_CPU_THREADS = None


def cpu_pick_threads():
    """Fastest thread count for a [2048,4096] x [4096,4096] fp32 matmul among powers of two."""
    global _CPU_THREADS
    if _CPU_THREADS is not None:
        return _CPU_THREADS
    import torch
    avail = len(os.sched_getaffinity(0))
    a = torch.randn(2048, 4096)
    b = torch.randn(4096, 4096)
    best, sweep = None, {}
    for t in [n for n in (8, 16, 32, 64, 128, 256) if n <= avail] or [avail]:
        torch.set_num_threads(t)
        a @ b
        ts = []
        for _ in range(3):
            t0 = time.perf_counter()
            a @ b
            ts.append(time.perf_counter() - t0)
        sweep[t] = round(sorted(ts)[1] * 1e3, 1)
        if best is None or sweep[t] < sweep[best] * 0.93:   # prefer fewer threads unless clearly faster
            best = t
    torch.set_num_threads(best)
    _CPU_THREADS = (best, sweep, avail)
    return _CPU_THREADS


class CpuSample:
    """Holds the tensors of the sample so that repeats time arithmetic, not allocation / RNG."""
    # 4096 = the workload's sequence length. The variable exists for the contract test of this arm (tests/
    # test_bench_reference_cpu.py); any other value is stated in the line's `sample` text.
    TOKENS = int(os.environ.get("B200W_BENCH_CPU_SAMPLE_TOKENS", "4096"))

    def __init__(self):
        import torch
        from oracle import llama_oracle as O
        self.torch, self.O = torch, O
        a = O.LLAMA2_7B
        self.a = a
        g = torch.Generator().manual_seed(0)
        one = O.Arch(a.vocab_size, a.hidden_size, a.intermediate_size, 1, a.num_heads, a.num_kv_heads,
                     a.head_dim, self.TOKENS, a.rms_norm_eps, a.rope_theta)
        shapes = O.param_shapes(one)
        self.layer = {k: (torch.randn(s, generator=g) * 0.02).requires_grad_(True) for k, s in shapes.items()
                      if k.startswith("model.layers.0.")}
        self.m = {k: torch.zeros_like(v) for k, v in self.layer.items()}
        self.v = {k: torch.zeros_like(v) for k, v in self.layer.items()}
        self.norm_w = torch.ones(a.hidden_size, requires_grad=True)
        self.head = (torch.randn(a.vocab_size, a.hidden_size, generator=g) * 0.02).requires_grad_(True)
        self.x = torch.randn(1, self.TOKENS, a.hidden_size, generator=g)
        self.labels = torch.randint(0, a.vocab_size, (1, self.TOKENS), generator=g)
        self.cos, self.sin = O.rope_cos_sin(self.TOKENS, a.head_dim, a.rope_theta)

    def run(self):
        """-> (seconds for the layer: fwd + bwd + AdamW, seconds for norm + lm_head + CE fwd + bwd)"""
        torch, O, a = self.torch, self.O, self.a
        import torch.nn.functional as F
        L, T = self.layer, self.TOKENS
        p = "model.layers.0."
        H, dh = a.num_heads, a.head_dim
        for w in list(L.values()) + [self.head, self.norm_w]:
            w.grad = None
        x = self.x.clone().requires_grad_(True)
        t0 = time.perf_counter()
        n = O.rmsnorm(x, L[p + "input_layernorm.weight"], a.rms_norm_eps)
        q = F.linear(n, L[p + "self_attn.q_proj.weight"]).view(1, T, H, dh).transpose(1, 2)
        k = F.linear(n, L[p + "self_attn.k_proj.weight"]).view(1, T, H, dh).transpose(1, 2)
        v = F.linear(n, L[p + "self_attn.v_proj.weight"]).view(1, T, H, dh).transpose(1, 2)
        q, k = O.apply_rope(q, self.cos, self.sin), O.apply_rope(k, self.cos, self.sin)
        # SDPA is what the HF path calls (sdpa_attention.py); the oracle's masked softmax is the same math
        o = F.scaled_dot_product_attention(q, k, v, is_causal=True).transpose(1, 2).reshape(1, T, H * dh)
        h = x + F.linear(o, L[p + "self_attn.o_proj.weight"])
        n2 = O.rmsnorm(h, L[p + "post_attention_layernorm.weight"], a.rms_norm_eps)
        h = h + O.swiglu_mlp(n2, L[p + "mlp.gate_proj.weight"], L[p + "mlp.up_proj.weight"],
                             L[p + "mlp.down_proj.weight"])
        t_fwd = time.perf_counter() - t0
        # the real loss on this layer's output: final norm, lm_head, HF causal-LM cross-entropy
        t0 = time.perf_counter()
        hd = h.detach().requires_grad_(True)
        loss, _ = O.causal_lm_loss(F.linear(O.rmsnorm(hd, self.norm_w, a.rms_norm_eps), self.head), self.labels,
                                   O.trainer_num_items(self.labels))
        loss.backward()
        t_head = time.perf_counter() - t0
        t0 = time.perf_counter()
        h.backward(hd.grad)
        with torch.no_grad():
            for kk, w in L.items():
                pn, mn, vn = O.adamw_update(w, w.grad, self.m[kk], self.v[kk], 1, 5e-5)
                w.copy_(pn); self.m[kk].copy_(mn); self.v[kk].copy_(vn)
        t_layer = t_fwd + time.perf_counter() - t0
        return t_layer, t_head


def cpu_measure(repeats: int, budget_s: float):
    """Median over `repeats` samples (at least 3; fewer only if one sample alone exceeds the budget).
    Returns (tokens/s of the full 32-layer step, description dict)."""
    threads, sweep, avail = cpu_pick_threads()
    smp = CpuSample()
    t0 = time.perf_counter()
    smp.run()                                   # warm-up: allocator, oneDNN primitive caches
    t_one = time.perf_counter() - t0
    n = max(3, min(repeats, int(budget_s / max(t_one, 1e-3))))
    if t_one > budget_s:
        n = 1
    t_runs = time.perf_counter()
    runs = [smp.run() for _ in range(n)]
    timed_wall = time.perf_counter() - t_runs
    a = smp.a
    per_seq = sorted(a.num_layers * tl + th for tl, th in runs)
    med = per_seq[len(per_seq) // 2]
    value = CpuSample.TOKENS / med
    desc = dict(value=round(value, 3), unit="tokens/s", cores=threads, kind="port",
                sample=(f"oracle port (fp32 torch, HF semantics): 1 of 32 true-width Llama-2-7B decoder layers "
                        f"fwd + bwd + AdamW on a full {CpuSample.TOKENS}-token sequence, plus final norm + lm_head + CE fwd/bwd "
                        f"(the real loss); step = 32 x layer + head per sequence, no extrapolation in tokens; "
                        f"median of {n} repeats after 1 warm-up"),
                repeats=n, spread_max_over_min=round(per_seq[-1] / per_seq[0], 3),
                layer_s=round(sorted(r[0] for r in runs)[n // 2], 3), head_s=round(sorted(r[1] for r in runs)[n // 2], 3),
                threads_sweep_ms=sweep, host_threads_available=avail,
                timed_wall_s=round(timed_wall, 2), warmup_wall_s=round(t_one, 2))
    return value, med, desc


def cpu_baseline(budget_s: float = 40.0):
    return cpu_measure(3, budget_s)[2]


def run_reference(args):
    """--impl reference: the reference's own path for this metric is the HF/PyTorch trainer
    image (un-vendored, examples/llama2-7b/finetuned-model.yaml:6); transformers.Trainer cannot
    be imported here (no `accelerate`), so its CPU path is the oracle port: same torch ops, host
    cores. Each step is the bounded sample of cpu_measure (one layer + head at full sequence
    length); at most ~4 minutes of samples are timed whatever --steps says, never fewer than 3."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    value, secs_per_seq, desc = cpu_measure(args.steps, 220.0)
    line = dict(impl="reference", metric=METRIC, value=round(value, 3), unit="tokens/s", n_gpus=args.gpus,
                steps=args.steps, warmup=args.warmup, ms_per_step=round(secs_per_seq * 1e3 * PER_DEVICE_BATCH, 1),
                higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f32", data="synthetic",
                config=workload_config(args.gpus), cpu_baseline=desc,
                e2e=dict(value=round(value, 3), unit="tokens/s", h2d_bytes_per_step=0,
                         d2h_bytes_per_step=0),
                # what a wall clock around this process sees is cpu_baseline.timed_wall_s (+ warm-up and imports), NOT
                # steps x ms_per_step: a step of this arm is a bounded SAMPLE (one of the 32 layers + the head, one of
                # the 8 sequences); ms_per_step is the full workload step that sample implies
                ms_per_step_is="32 x layer_s + head_s per sequence, x 8 sequences (cpu_baseline.layer_s / head_s); "
                               "wall time actually spent: cpu_baseline.timed_wall_s")
    emit(line)


PER_DEVICE_BATCH = 8


RECOMPUTE = False
MICRO_BATCH = 2   # sequences per accumulation micro-step: T = 8192 rows per GEMM (see workload_config)
SHARD_STATE = False
def gemm_traffic():
    """DRAM bytes per launch of the dominant kernel from the committed `ncu --set full` capture of THIS kernel
    family at THIS micro-batch's shape (profiles/r02_ncu_gemm_mb2_banded.json for M = 8192 tokens, r02_ncu_gemm.json
    for M = 4096; written from the .ncu-rep by tools/ncu_gemm_json.py): the forward gate|up GEMM, with the dgrad and
    accumulating-wgrad captures beside it."""
    name = "r02_ncu_gemm_mb2_banded.json" if MICRO_BATCH == 2 else "r02_ncu_gemm.json"
    path = os.path.join(ROOT, "profiles", name)
    try:
        j = json.load(open(path))
        d = j["kernels"]
        f = d["fwd_gateup"]
        return dict(bytes=f["dram_read_bytes"] + f["dram_write_bytes"],
                    note=(f"dram__bytes_read+write of one forward gate|up GEMM launch (M{j.get('tokens', 4096)} N22016 K4096) = "
                          f"{f['traffic_over_algorithmic']}x its {f['algorithmic_bytes'] / 1e6:.0f} MB algorithmic; dgrad "
                          f"{d['dgrad_gateup']['traffic_over_algorithmic']}x, accumulating wgrad "
                          f"{d['wgrad_gateup_acc']['traffic_over_algorithmic']}x (profiles/{name}, ncu --set full)"))
    except Exception:  # noqa: BLE001
        return dict(bytes=None, note=f"profiles/{name} missing")


DUMP_SAMPLE = 65536   # elements kept per weight matrix by --dump-outputs


def dump_outputs(out_dir: str, e, loss: float, grad_norm: float):
    """What the last timed step returns to its caller: loss and grad-norm, and the fp32 master weights it
    updated -- of the first and last decoder layers and every tensor outside the layers (embedding, final
    norm, lm_head). A matrix is kept as DUMP_SAMPLE elements at fixed seeded flat indices, a vector whole:
    4.3 MB in all at Llama-2-7B size. Each array goes to out_dir/<name>.npy."""
    import numpy as np

    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "loss.npy"), np.float64(loss))
    np.save(os.path.join(out_dir, "grad_norm.npy"), np.float64(grad_norm))
    keep = (".layers.0.", f".layers.{e.arch.num_layers - 1}.")
    for i, (name, shape) in enumerate(e.params()):
        if ".layers." in name and not any(k in name for k in keep):
            continue
        w = e.read_state(name, shape, "master").reshape(-1)
        if len(shape) > 1 and w.size > DUMP_SAMPLE:
            w = w[np.sort(np.random.default_rng(i).choice(w.size, DUMP_SAMPLE, replace=False))]
        np.save(os.path.join(out_dir, name + ".npy"), w)


def workload_config(n_gpus: int):
    return dict(workload="Llama-2-7B bf16 causal-LM fine-tune, seq 4096 (BASELINE.json configs[1])",
                global_batch=PER_DEVICE_BATCH * n_gpus, seq_len=4096, per_device_batch=PER_DEVICE_BATCH,
                micro_batch=MICRO_BATCH, parallelism=f"dp{n_gpus}" + ("-sharded-state" if SHARD_STATE and n_gpus > 1 else ""),
                optimizer="AdamW fp32 master, clip 1.0" + (", activation recomputation" if RECOMPUTE else ""),
                l2="working set (13.5 GB bf16 weights + activations per micro-step) >> 126 MB L2; no flush needed",
                micro_batch_note=("the per-device batch of 8 sequences runs as 4 accumulation micro-steps of 2: the N = 4096 "
                                  "GEMMs then have 512 instead of 256 output tiles for 74 CTA pairs (98.8 % instead of 86.5 % wave "
                                  "efficiency); same arithmetic as 8 x 1 (tests/test_engine.py 'accumulate' vs 'full')"))


# --------------------------------------------------------------------------------------------
# the CUDA arm
# --------------------------------------------------------------------------------------------
def run_ours(args):
    import numpy as np
    import torch

    from runbooks_b200.engine import Engine, LlamaArch

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch N>1 with torch.distributed.run (one rank per GPU)")
    dist = None
    if world > 1:
        import torch.distributed as dist_
        dist = dist_
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("gloo", rank=rank, world_size=world)  # control plane only
    torch.cuda.set_device(local)
    # The decode metric runs FIRST (its engine is destroyed before the fine-tune model is built): each leg is an
    # independent measurement, and after ~40 s of fine-tune steps at the 1 kW power cap the decode leg read 1.7 %
    # lower than alone (profiles/r02_decode_v4_tiled.json vs the embedded object of r02_bench_n1_v14.json).
    decode_obj = None
    if world == 1 and not args.no_decode:
        try:
            decode_obj = decode_leg(local)
        except Exception as ex:  # noqa: BLE001 -- the fine-tune line must not be lost to the second metric
            decode_obj = dict(error=f"{type(ex).__name__}: {ex}")
        torch.cuda.empty_cache()
    arch = LlamaArch.llama2_7b(4096)
    if args.layers:  # development knob; a reduced model is NOT the benchmark and is labelled so
        arch.num_layers = args.layers
    S, nseq = arch.max_seq_len, args.per_device_batch
    e = Engine(local)
    shard = bool(args.shard_state) and world > 1
    uid = None
    if world > 1:
        uid = torch.zeros(128, dtype=torch.uint8)
        if rank == 0:
            uid = torch.frombuffer(bytearray(e.comm_unique_id()), dtype=torch.uint8).clone()
        dist.broadcast(uid, 0)
        uid = bytes(uid.numpy().tobytes())
    if shard:                                # sharded optimiser state: the communicator comes first
        e.comm_init(rank, world, uid)
    e.init_model(arch, micro_batch=args.micro_batch, training=True, shard_state=shard, recompute=bool(args.recompute))
    e.init_random(seed=0, std=0.02)          # identical replicas: same seed on every rank
    if world > 1 and not shard:
        e.comm_init(rank, world, uid)

    g = torch.Generator().manual_seed(1234 + rank)
    n_prof = min(args.steps, 3)               # GEMM-bracketed steps for the roofline leg, outside both timed regions
    # every step of every region sees a FRESH batch: a 7B model memorises a 32k-token batch of random ids
    # after one exposure (round 1's e2e region re-used the resident region's batches and printed loss 2.7
    # where fresh uniform tokens cannot go below ln 32000 = 10.4)
    n_batches = args.warmup + 2 * args.steps + n_prof
    host_ids = torch.randint(0, arch.vocab_size, (n_batches, nseq, S), generator=g, dtype=torch.int32).pin_memory()
    dev_ids = host_ids[: args.warmup + args.steps].cuda()
    n_valid = nseq * S                        # HF Trainer's num_items_in_batch: labels = ids, none ignored
    tokens_per_step = nseq * S

    def require_finite(where, loss_v, gn_v):
        # NaN operands toggle no tensor-core inputs: the chip leaves its power cap and the step
        # "speeds up". Such a run is not a measurement; fail loudly instead of printing a number.
        # (loss / grad-norm are global values, identical on every rank, so all ranks stop together)
        if not (math.isfinite(loss_v) and math.isfinite(gn_v)):
            raise SystemExit(f"bench.py: {where}: loss={loss_v} grad_norm={gn_v} not finite; no result printed")

    def barrier():
        e.sync()
        torch.cuda.synchronize()
        if dist:
            dist.barrier()

    # ---- warm-up (host API: also exercises the e2e path) ----
    for i in range(args.warmup):
        ids = host_ids[i].numpy()
        loss, gn = e.train_step(ids, ids, lr=5e-5)
    require_finite("warm-up", loss, gn)
    barrier()

    # ---- timed region 1: inputs resident in HBM ----
    launches0 = e.launch_count()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    barrier()
    e.timer_start()
    for i in range(args.steps):
        p = dev_ids[args.warmup + i].data_ptr()
        e.train_step_resident(p, p, nseq, n_valid, lr=5e-5)
    ms = e.timer_stop()
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    launches = e.launch_count() - launches0
    loss_res, gn_res = e.read_scalars()
    require_finite("resident timed region", loss_res, gn_res)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, e, loss_res, gn_res)

    # ---- timed region 2: end to end through the host-buffer API ----
    barrier()
    e.timer_start()
    t_wall = time.perf_counter()
    for i in range(args.steps):
        ids = host_ids[args.warmup + args.steps + i].numpy()
        loss, gn = e.train_step(ids, ids, lr=5e-5)   # H2D of ids+labels, D2H of loss/grad-norm inside
    ms_e2e = e.timer_stop()
    wall_e2e = (time.perf_counter() - t_wall) * 1e3
    require_finite("e2e timed region", loss, gn)
    barrier()
    ms_e2e = max(ms_e2e, wall_e2e)  # host-side work (pinned staging, sync) counts end to end

    # ---- roofline leg: the same step with every GEMM launch bracketed by CUDA events. Kept OUT of the
    # regions that produce `value` and `e2e` (the 2 x 774 event records per micro-step cost ~0.6 %) ----
    e.profile_gemm(True)
    e.timer_start()
    for i in range(n_prof):
        ids = host_ids[args.warmup + 2 * args.steps + i].numpy()
        e.train_step(ids, ids, lr=5e-5)
    ms_prof = e.timer_stop()
    gemm_ms, gemm_flops, gemm_launches = e.profile_read()
    e.profile_gemm(False)
    barrier()

    per_rank = None
    if dist:
        # every rank's own GEMM rate in the bracketed steps: the ranks move in lock-step (each all-reduce waits
        # for the slowest), so the spread of these rates is what a data-parallel step loses to the slowest GPU
        mine = torch.tensor([gemm_flops / (gemm_ms / 1e3) / 1e12 if gemm_ms > 0 else 0.0, ms], dtype=torch.float64)
        allr = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(allr, mine)
        per_rank = dict(gemm_tflops=[round(float(x[0]), 1) for x in allr],
                        resident_ms_per_step=[round(float(x[1]) / args.steps, 2) for x in allr])
        t = torch.tensor([ms, ms_e2e], dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, ms_e2e = float(t[0]), float(t[1])
    if rank != 0:
        return
    pk = peaks()
    total_tokens = tokens_per_step * world * args.steps
    value = total_tokens / (ms / 1e3)
    e2e = total_tokens / (ms_e2e / 1e3)
    achieved = gemm_flops / (gemm_ms / 1e3) / 1e12 if gemm_ms > 0 else None
    cfg = workload_config(world)
    if args.layers:
        cfg["workload"] += f" — REDUCED to {args.layers} layers (development run, not the benchmark)"
    line = dict(
        metric=METRIC, value=round(value, 1), unit="tokens/s", n_gpus=world, steps=args.steps,
        warmup=args.warmup, ms_per_step=round(ms / args.steps, 2), higher_is_better=True, scaling="weak",
        vs_baseline=None, dtype="bf16", data="synthetic", config=cfg,
        e2e=dict(value=round(e2e, 1), unit="tokens/s", h2d_bytes_per_step=2 * tokens_per_step * 4,
                 d2h_bytes_per_step=16),
        gpu_launches=int(launches),
        roofline=dict(bound="tensor", achieved=round(achieved, 1) if achieved else None,
                      peak=pk["sustained"], unit="TFLOP/s",
                      frac=round(achieved / pk["sustained"], 4) if achieved else None,
                      # DRAM bytes of ONE launch (gate|up forward, M4096 N22016 K4096) read from the committed
                      # `ncu --set full` capture; its algorithmic bytes are 394 MB (A 33.5 + B 180.4 + D 180.4)
                      traffic=gemm_traffic()["bytes"], traffic_note=gemm_traffic()["note"],
                      kernel="gemm_bf16_kernel (tcgen05)", launches=int(gemm_launches),
                      share_of_step=round(gemm_ms / ms_prof, 4), profiled_steps=n_prof,
                      peak_source=f"{pk['source']} sustained cuBLAS bf16 (kernel timed inside a long step)"),
        model_flops=dict(per_token=FLOPS_PER_TOKEN,
                         achieved_tflops_per_gpu=round(value / world * FLOPS_PER_TOKEN / 1e12, 1),
                         frac_of_sustained_peak=round(value / world * FLOPS_PER_TOKEN / 1e12 / pk["sustained"], 4),
                         frac_of_burst_peak=round(value / world * FLOPS_PER_TOKEN / 1e12 / pk["burst"], 4)),
        clocks=clocks, loss=round(float(loss), 4), grad_norm=round(float(gn), 4),
        device_gb=round(e.device_bytes() / 1e9, 1),
    )
    if per_rank:
        line["per_rank"] = per_rank
    e.close()
    if decode_obj is not None:
        line["decode"] = decode_obj
    if world == 1 and not args.no_cpu:
        line["cpu_baseline"] = cpu_baseline()
    emit(line)


# --------------------------------------------------------------------------------------------
# decode leg (BASELINE.json configs[3], SURVEY.md 8d second metric): Falcon-7B-Instruct layout,
# random-init bf16 weights, batch 32, context 1024, greedy, through b200w_infer_step with HOST buffers
# --------------------------------------------------------------------------------------------
def decode_leg(device: int = 0, batch: int = 32, ctx: int = 1024, steps: int = 64, warm: int = 4):
    import numpy as np

    from runbooks_b200.infer import InferEngine, ServeArch

    arch = ServeArch.falcon_7b(max_ctx=ctx + steps + warm + 8)
    e = InferEngine(device)
    e.init_infer(arch, max_batch=batch)
    e.infer_init_random(0, 0.02)
    rng = np.random.default_rng(0)
    slots = list(range(batch))
    prompts = rng.integers(0, arch.vocab_size, size=(batch, ctx)).tolist()
    # the context is built by the one-pass prefill (also timed: it is the other half of serving a request)
    chunk = 8                                  # 8 x 1024 tokens per prefill call
    e.prefill(prompts[:chunk], slots[:chunk])  # warm-up (buffer growth, first-use attributes)
    e.sync()
    t0 = time.perf_counter()
    tok = []
    for i in range(0, batch, chunk):
        nxt, _ = e.prefill(prompts[i:i + chunk], slots[i:i + chunk])
        tok.extend(int(t) for t in nxt)
    e.sync()
    prefill_s = time.perf_counter() - t0
    tok = np.array(tok, dtype=np.int32)
    for w in range(warm):                      # eager run, graph capture, replays
        tok, _ = e.step(tok, [ctx + w] * batch, slots)
    e.sync()
    if os.environ.get("B200W_PROFILE_DECODE"):   # ncu --profile-from-start off: exactly two decode steps
        import torch
        torch.cuda.profiler.start()
        for i in range(2):
            e.step(tok, [ctx + warm] * batch, slots)
        torch.cuda.profiler.stop()
    launches0 = e.launch_count()
    e.timer_start()
    t0 = time.perf_counter()
    for i in range(steps):
        tok, _ = e.step(tok, [ctx + warm + i] * batch, slots)   # H2D of 3 x 32 ints, D2H of 32 ints inside
    ms = e.timer_stop()
    wall = (time.perf_counter() - t0) * 1e3
    launches = e.launch_count() - launches0
    n_params = sum(int(np.prod(s)) for _, s in e.infer_params())
    kv_bytes = batch * (ctx + warm + steps // 2) * arch.num_layers * 2 * arch.num_kv_heads * arch.head_dim * 2
    bytes_step = 2 * n_params + kv_bytes
    pk = peaks()
    per = max(ms, wall) / steps
    e.close()
    return dict(
        metric="Falcon-7B greedy decode tokens/s, batch 32, context 1024, 1xB200 (BASELINE.json configs[3])",
        value=round(batch / (per / 1e3), 1), unit="tokens/s", ms_per_step=round(per, 3),
        device_ms_per_step=round(ms / steps, 3), steps=steps, dtype="bf16", data="synthetic (random-init weights, random prompts)",
        e2e=dict(value=round(batch / (wall / steps / 1e3), 1), unit="tokens/s", h2d_bytes_per_step=3 * batch * 4,
                 d2h_bytes_per_step=batch * 4),
        gpu_launches_per_step=round(launches / steps, 1),
        roofline=dict(bound="hbm", achieved=round(bytes_step / (per / 1e3) / 1e9, 1), peak=pk["hbm"], unit="GB/s",
                      frac=round(bytes_step / (per / 1e3) / 1e9 / pk["hbm"], 4), traffic=None,
                      algorithmic_bytes_per_step=int(bytes_step), params=n_params,
                      note="bytes = 2 x parameters (every weight read once per step, the tied embedding as lm_head) "
                           "+ K/V of batch x context; peak = measured copy bandwidth (MEASURED_PEAKS.json)"),
        prefill=dict(tokens=batch * ctx, seconds=round(prefill_s, 3), tokens_per_s=round(batch * ctx / prefill_s, 1),
                     note="one-pass prompt ingestion (b200w_infer_prefill), 4 calls of 8 x 1024 tokens"))


_REAL_STDOUT = None


def claim_stdout():
    """The contract is ONE JSON line on stdout. Libraries write there too (NCCL prints its version
    banner with printf), so fd 1 is pointed at stderr for the whole run and the JSON line goes to
    the saved original."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def emit(line: dict):
    out = _REAL_STDOUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def main():
    global MICRO_BATCH, SHARD_STATE, RECOMPUTE
    claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=4)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--per-device-batch", type=int, default=PER_DEVICE_BATCH)
    ap.add_argument("--micro-batch", type=int, default=MICRO_BATCH,
                    help="sequences per accumulation micro-step (activation memory scales with it)")
    ap.add_argument("--layers", type=int, default=0, help="development only: fewer layers")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-decode", action="store_true", help="skip the Falcon-7B decode leg (N=1 only)")
    ap.add_argument("--recompute", action="store_true",
                    help="activation recomputation (NOT the benchmark default: the extra forward work is real work "
                         "but not algorithmic FLOPs; the line is labelled)")
    ap.add_argument("--shard-state", action="store_true", default=bool(os.environ.get("B200W_SHARD_STATE")),
                    help="N>1: fp32 master / Adam moments sharded over the ranks (reduce-scatter + all-gather)")
    ap.add_argument("--decode-only", action="store_true", help="run only the decode leg and print its object")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed fine-tune step computed (loss, grad-norm, sampled updated "
                         "weights) as DIR/<name>.npy; the inputs depend only on the arguments")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "ours" or args.decode_only):
        ap.error("--dump-outputs writes the outputs of the CUDA fine-tune step (--impl ours, not --decode-only)")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    MICRO_BATCH = args.micro_batch
    RECOMPUTE = bool(args.recompute)
    SHARD_STATE = bool(args.shard_state)
    # A rank that fails must EXIT, at once: its peers are inside a collective that can no longer
    # complete, and the launcher only tears the job down when a worker process ends. Interpreter
    # teardown (destructors -> NCCL / CUDA shutdown on a dead context) can block, so skip it.
    # (profiles/r01_n8_failure.txt: one rank raised, did not exit, and 7 GPUs spun for 10 minutes.)
    code = 0
    try:
        if args.decode_only:
            emit(decode_leg(int(os.environ.get("LOCAL_RANK", "0"))))
        elif args.impl == "reference":
            run_reference(args)
        else:
            run_ours(args)
    except SystemExit as ex:
        code = ex.code if isinstance(ex.code, int) else 1
        if not isinstance(ex.code, int) and ex.code is not None:
            sys.stderr.write(str(ex.code) + "\n")
    except BaseException:  # noqa: BLE001
        import traceback
        traceback.print_exc()
        code = 1
    finally:
        for f in (sys.stderr, _REAL_STDOUT, sys.stdout):
            try:
                if f:
                    f.flush()
            except Exception:  # noqa: BLE001
                pass
    if code:
        os._exit(code)


if __name__ == "__main__":
    main()
