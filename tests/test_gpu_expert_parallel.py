"""Expert-parallel MoE (SURVEY.md 8e) with the real kernels: each rank owns the experts e % world == rank of a small Mixtral-style
model; the down projection's epilogue stores every weighted expert row into every rank's row buffer (CUDA-IPC peer memory), a
flag handshake follows, and every rank combines all rows in the reference's order (csrc/moe.cuh).  Prefill + decode logits must
equal the UNSHARDED model's bit for bit -- for top-2 and for top-3 routing (no reduction order is left open).

Two set-ups:
  * two processes sharing cuda:0 (gloo for the handle exchange): one GPU is enough, peer stores go through IPC mappings of the
    same device; the handshake spins across time slices, so it is slow but exercises the whole protocol;
  * one process per GPU with NCCL (needs >= 2 GPUs; skipped on a one-GPU machine): peer stores cross NVLink.
"""
import os
import socket
import sys
from pathlib import Path

import pytest
import torch
import torch.multiprocessing as mp

REPO = Path(__file__).resolve().parents[1]
pytestmark = pytest.mark.gpu


def _free_port() -> int:
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank: int, world: int, port: int, q, backend: str, top_k: int):
    try:
        sys.path.insert(0, str(REPO))
        os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
        dev = rank if backend == "nccl" else 0
        torch.cuda.set_device(dev)
        if backend == "nccl":
            torch.distributed.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", dev))
        else:
            torch.distributed.init_process_group("gloo", rank=rank, world_size=world)
        import mistral_inference_b200 as mi
        import synth
        from mistral_inference_b200.cache import BufferCache
        from mistral_inference_b200.transformer import Transformer

        p = synth.shape("tiny-moe", sliding_window=16)
        p["moe"] = dict(p["moe"], num_experts_per_tok=top_k)
        sd = synth.synth_state_dict(p, 2, torch.bfloat16, "cuda")

        def build(expert_parallel):
            args = mi.TransformerArgs.from_dict(dict(p))
            args.max_batch_size = 2
            m = Transformer.empty(args, "cuda", torch.bfloat16, expert_parallel=expert_parallel)
            m.load_state_dict(sd)
            return m.eval()

        def run(m):
            cache = BufferCache(m.n_local_layers, 2, 64, p["n_kv_heads"], p["head_dim"], p.get("sliding_window")).to(m.device, m.dtype)
            seqlens = [12, 9]
            toks = torch.tensor(synth.synth_prompt(sum(seqlens), p["vocab_size"], 4), device="cuda")
            outs = [m.forward(toks, seqlens, cache)]
            nxt = torch.tensor([5, 7], device="cuda")
            for _ in range(4):  # eager warm-up, graph capture, graph replays
                lg = m.forward(nxt, [1, 1], cache)
                outs.append(lg)
                nxt = lg.argmax(-1)
            return torch.cat(outs).cpu()

        sharded = run(build((rank, world)))  # both ranks run in lock step: the handshakes pair up
        torch.distributed.barrier()
        full = run(build(None)) if rank == 0 else None
        ok = bool(torch.equal(sharded, full)) if rank == 0 else True
        worst = float((sharded - full).abs().max()) if rank == 0 else 0.0
        q.put((rank, ok, worst, ""))
        torch.distributed.barrier()
        torch.distributed.destroy_process_group()
    except Exception as e:  # surface the failure in the parent instead of a queue timeout
        q.put((rank, False, -1.0, repr(e)))
        raise


def _run(backend: str, top_k: int):
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q, backend, top_k)) for r in range(2)]
    for pr in procs:
        pr.start()
    res = sorted(q.get(timeout=400) for _ in range(2))
    for pr in procs:
        pr.join(timeout=60)
    for rank, ok, worst, err in res:
        assert ok, f"rank {rank}: {err or 'sharded logits differ from the unsharded model by %g' % worst}"
    assert all(pr.exitcode == 0 for pr in procs)


@pytest.mark.parametrize("top_k", [2, 3])
def test_expert_parallel_equals_unsharded_two_processes_one_gpu(top_k):
    _run("gloo", top_k)


@pytest.mark.parametrize("top_k", [2, 3])
def test_expert_parallel_equals_unsharded_two_gpus_nccl(top_k):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    _run("nccl", top_k)


# ----------------------------------------------------------------------------- reference-compatible pipeline mode on GPUs
# (needs two GPUs: the pipeline's send / recv / broadcast of CUDA tensors is NCCL's job -- gloo cannot send device memory, and NCCL
# refuses two ranks on one device)
def _pp_worker(rank: int, world: int, port: int, q, backend: str):
    try:
        sys.path.insert(0, str(REPO))
        os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
        dev = rank if backend == "nccl" else 0
        torch.cuda.set_device(dev)
        if backend == "nccl":
            torch.distributed.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", dev))
        else:
            torch.distributed.init_process_group("gloo", rank=rank, world_size=world)
        import mistral_inference_b200 as mi
        import synth
        from mistral_inference_b200.transformer import Transformer

        p = synth.shape("tiny", n_layers=4, sliding_window=16)
        sd = synth.synth_state_dict(p, 2, torch.bfloat16, "cuda")
        args = mi.TransformerArgs.from_dict(dict(p))
        args.max_batch_size = 2
        prompts = [synth.synth_prompt(12, p["vocab_size"], 4), synth.synth_prompt(9, p["vocab_size"], 5)]
        m = Transformer.empty(args, "cuda", torch.bfloat16, pipeline_rank=rank, num_pipeline_ranks=world)
        m.load_state_dict(sd)
        toks, lp = mi.generate(prompts, m.eval(), max_tokens=5, temperature=0.0)  # transformer.py:188-237: send / recv / broadcast
        torch.distributed.barrier()
        ok, err = True, ""
        if rank == 0:
            full = Transformer.empty(args, "cuda", torch.bfloat16)
            full.load_state_dict(sd)
            t2, lp2 = mi.generate(prompts, full.eval(), max_tokens=5, temperature=0.0)
            worst = max(abs(a - b) for x, y in zip(lp, lp2) for a, b in zip(x, y))
            ok = toks == t2 and worst <= 0.03  # the pipeline's lm head is a bf16 Linear + .float() (transformer.py:235-240), like the single-stage path
            err = f"tokens {toks} vs {t2}, max|d logprob| {worst}"
        q.put((rank, ok, 0.0, "" if ok else err))
        torch.distributed.barrier()
        torch.distributed.destroy_process_group()
    except Exception as e:
        q.put((rank, False, -1.0, repr(e)))
        raise


def _run_pp(backend: str):
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_pp_worker, args=(r, 2, port, q, backend)) for r in range(2)]
    for pr in procs:
        pr.start()
    res = sorted(q.get(timeout=400) for _ in range(2))
    for pr in procs:
        pr.join(timeout=60)
    for rank, ok, _, err in res:
        assert ok, f"rank {rank}: {err}"
    assert all(pr.exitcode == 0 for pr in procs)


def test_pipeline_ranks_two_gpus_nccl():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    _run_pp("nccl")
