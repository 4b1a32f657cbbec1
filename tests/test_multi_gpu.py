"""Multi-GPU parity inside `pytest -m gpu` (the two-rank tests skip on a machine with fewer than 2 GPUs).

  * two ranks, one process each, NCCL communicator through the C ABI: after the data-parallel step the
    ranks' weights are BIT-IDENTICAL, and equal to the single-GPU step on the whole global batch within
    1e-3 (bf16 wire format of the gradient all-reduce: SURVEY.md 8 a11 / e);
  * the overlapped per-matrix all-reduce (default) and the one-shot all-reduce after the backward
    (B200W_AR_MODE=end) give the same weights bit for bit;
  * one process holding contexts on two devices (the cgo host model of INTEGRATION.md): per-device
    function attributes and SM counts (round 1 cached them per process).
Oracle for the arithmetic: tests/test_data_parallel_cpu.py pins the formulation (sum of per-rank
sum(nll) / n_global == single process on the concatenated batch) against HF's loss on CPU/gloo."""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _gpus():
    import torch
    return torch.cuda.device_count()


def _rank_main(rank, world, uid, q, mode, steps, comm1=False):
    try:
        shard = mode == "shard"
        if mode and not shard:
            os.environ["B200W_AR_MODE"] = mode
        import sys
        root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
        for p in (root, os.path.join(root, "tests")):
            if p not in sys.path:
                sys.path.insert(0, p)
        from oracle import llama_oracle as O
        from runbooks_b200.engine import Engine, LlamaArch
        fx = np.load(os.path.join(root, "tests", "golden", "llama_tiny_mha.npz"))
        v = [int(x) for x in fx["arch"]]
        eps, theta = (float(x) for x in fx["arch_f"])
        oa = O.Arch(*v, rms_norm_eps=eps, rope_theta=theta)
        params = O.seeded_params(oa, int(fx["batch"][1]))
        e = Engine(rank)
        want_comm = world > 1 or comm1     # comm1: a ONE-rank communicator (the exchange path on a 1-GPU box)
        if want_comm and shard:
            e.comm_init(rank, world, uid)          # sharded state: the communicator comes first
        e.init_model(LlamaArch(*v, rms_norm_eps=eps, rope_theta=theta), micro_batch=1, training=True,
                     shard_state=shard)
        e.load_state_dict(params)
        if want_comm and not shard:
            e.comm_init(rank, world, uid)
        out = []
        for ids, labels, lr in ((fx["ids"], fx["labels"], 5e-5), (fx["ids2"], fx["labels2"], 2.5e-5))[:steps]:
            # make the ranks hold DIFFERENT numbers of targets: the normaliser must be the global count
            labels = labels.copy()
            labels[1, 40:90] = -100
            mine = slice(rank, None, world)
            out.append(e.train_step(ids[mine], labels[mine], lr=lr))
        sd = {n: (e.read_tensor(n, s, bf16_bits=True) if mode in ("shard", "bits") else e.read_state(n, s, "master"))
              for n, s in e.params()}
        q.put((rank, out, sd, None))
        e.close()
    except BaseException as ex:  # noqa: BLE001
        import traceback
        q.put((rank, None, None, traceback.format_exc()))
        os._exit(1)


def _run(world, mode=None, steps=2, comm1=False):
    import multiprocessing as mp
    from runbooks_b200.engine import Engine
    uid = b""
    if world > 1 or comm1:
        e = Engine(0)
        uid = e.comm_unique_id()
        e.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_rank_main, args=(r, world, uid, q, mode, steps, comm1)) for r in range(world)]
    for p in procs:
        p.start()
    res = {}
    for _ in range(world):
        rank, out, sd, err = q.get(timeout=300)
        assert err is None, f"rank {rank} failed:\n{err}"
        res[rank] = (out, sd)
    for p in procs:
        p.join(60)
    return res


@pytest.mark.skipif(_gpus() < 2, reason="needs 2 GPUs")
def test_two_ranks_are_bit_identical_and_match_one_gpu():
    two = _run(2)
    one = _run(1)
    (out0, sd0), (out1, sd1) = two[0], two[1]
    assert out0 == out1, (out0, out1)                      # global loss / grad-norm: the same floats on both ranks
    for n in sd0:
        assert np.array_equal(sd0[n], sd1[n]), f"ranks diverged on {n}"
    out_one, sd_one = one[0]
    for (l2, g2), (l1, g1) in zip(out0, out_one):
        assert abs(l2 - l1) < 1e-4 * abs(l1) and abs(g2 - g1) < 2e-3 * g1, (out0, out_one)
    worst = max(float(np.linalg.norm(sd0[n] - sd_one[n]) / np.linalg.norm(sd_one[n])) for n in sd0)
    print(f"1-GPU vs 2-GPU updated weights: worst relative difference {worst:.3e}")
    assert worst < 1e-3


def test_one_rank_communicator_overlap_equals_end_bit_for_bit():
    """Runs on a 1-GPU box: a one-rank NCCL communicator drives the whole exchange path. In overlap mode the last
    micro-step's wgrad GEMMs write the bf16 wire copy from their epilogue (gemm.cu EpiExtra::d2) and no cast
    pass runs for those ranges; in `end` mode a cast kernel rounds the fp32 sum afterwards. Same rounding of the
    same fp32 value: the updated weights must agree bit for bit (2 accumulation micro-steps per step)."""
    a = _run(1, "overlap", steps=2, comm1=True)
    b = _run(1, "end", steps=2, comm1=True)
    assert a[0][0] == b[0][0]
    for n in a[0][1]:
        assert np.array_equal(a[0][1][n], b[0][1][n]), n


@pytest.mark.skipif(_gpus() < 2, reason="needs 2 GPUs")
def test_overlapped_and_end_allreduce_agree_bit_for_bit():
    a = _run(2, "overlap", steps=1)
    b = _run(2, "end", steps=1)
    for n in a[0][1]:
        assert np.array_equal(a[0][1][n], b[0][1][n]), n


@pytest.mark.skipif(_gpus() < 2, reason="needs 2 GPUs")
def test_sharded_optimizer_state_equals_replicated():
    """b200w_model_init(training = 2): reduce-scatter -> AdamW on the owned 1/N of master / m / v -> all-gather
    of the bf16 weights (SURVEY.md 8e, the 70B row's groundwork). At two ranks a sum of two terms has one
    order, so the weights must equal the replicated mode's bit for bit; ranks agree with each other."""
    a = _run(2, "shard")
    b = _run(2, "bits")
    assert a[0][0] == a[1][0] and a[0][0] == b[0][0], (a[0][0], b[0][0])      # loss / grad-norm
    for n in a[0][1]:
        assert np.array_equal(a[0][1][n], a[1][1][n]), f"ranks diverged on {n}"
        assert np.array_equal(a[0][1][n], b[0][1][n]), f"sharded != replicated on {n}"


@pytest.mark.skipif(_gpus() < 2, reason="needs 2 GPUs")
def test_one_process_two_devices():
    """INTEGRATION.md's cgo layout: one host process, one context per device, driven from one thread here.
    The > 48 KB dynamic-shared-memory attribute of every kernel must be set on BOTH devices."""
    import torch
    from runbooks_b200.engine import Engine
    from util import call, rel_err
    outs = []
    for dev_i in (0, 1):
        e = Engine(dev_i)
        with torch.cuda.device(dev_i):
            g = torch.Generator().manual_seed(3)
            A = torch.randn(512, 256, generator=g).bfloat16().cuda()
            B = torch.randn(512, 256, generator=g).bfloat16().cuda()
            D = torch.empty(512, 512, device="cuda", dtype=torch.bfloat16)
            call(e, "b200w_op_gemm", A, 0, 256, B, 0, 256, D, None, 0, 512, 512, 512, 256, 512)   # CTA-pair kernel
            S, H = 256, 2
            qkv = torch.randn(S, 3 * H * 128, generator=g).bfloat16().cuda()
            o = torch.empty(S, H * 128, device="cuda", dtype=torch.bfloat16)
            lse = torch.empty(H, S, device="cuda", dtype=torch.float32)
            call(e, "b200w_op_attention_fwd", qkv, 3 * H * 128, H * 128, 2 * H * 128, o, H * 128, lse, 1, S, H, H,
                 128 ** -0.5)
            torch.cuda.synchronize()
            assert rel_err(D.float().cpu(), A.float().cpu() @ B.float().cpu().T) < 5e-3
            outs.append((D.cpu(), o.cpu()))
        e.close()
    assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1])
