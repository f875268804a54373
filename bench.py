#!/usr/bin/env python
"""bench.py -- BASELINE.json metric: decode tokens/s (bf16, batch=1, 4k context) + prefill TFLOPS vs roofline.

Default workload = BASELINE.json configs[1]: Mistral-7B full (32 layers, GQA 32/8, sliding_window=4096), random-init bf16,
1xB200, batch 1, 4096-token prefill, then decode.  A "step" = one decode step (one pass of the hot path over the batch).

    python bench.py --gpus N --steps K --warmup W              # this repo's CUDA path
    python bench.py --impl reference --gpus N ...               # the reference's algorithm on the host CPUs (full depth)
    python bench.py --model mistral-nemo-12b --batch 32 --prefill 1024    # BASELINE configs[2] (informational lines)
    python bench.py --gpus 1 --steps K --warmup W --dump-outputs DIR      # + the last timed step's outputs as DIR/*.npy
    torchrun ... bench.py --gpus N --parallel expert --model mixtral-8x7b --batch 8 --prefill 2048   # configs[3]/[4]: expert-sharded

Under torchrun (N > 1) the dense 7B model is "replicas only" (it fits one GPU; DESIGN.md section (e)): every rank runs the same
workload, value = N * B * K / max-over-ranks time, scaling "weak"; the line then also carries a `sharded` sub-record: the
expert-parallel Mixtral decode step (the path's one real exchange) measured on the same N GPUs.

Prints ONE JSON line.  Timing: CUDA events on the launching stream, W >= 3 warm-up steps, inputs (>= 14 GB of weights per step)
far larger than the 126 MB L2.
"""
import argparse
import json
import math
import os
import shutil
import statistics
import subprocess
import sys
import threading
import time
from pathlib import Path

import torch

REPO = Path(__file__).resolve().parent
sys.path.insert(0, str(REPO))

import synth  # noqa: E402

METRIC = "decode tokens/sec (bf16, batch=1, seq=4k) [+ prefill TFLOPS, both vs roofline]"


# ------------------------------------------------------------------------------------------------ helpers
def measured_peaks():
    f = REPO / "MEASURED_PEAKS.json"
    if f.exists():
        d = json.loads(f.read_text())
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"], "bf16_tflops_sustained": d.get("bf16_tflops_sustained"),
                "source": "measured (MEASURED_PEAKS.json)"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback (B200_PROFILING.md)"}


def experts_touched(E: int, k: int, batch: int) -> float:
    """Expected number of distinct experts a layer streams for `batch` tokens under uniform routing (SURVEY.md 8d)."""
    return E * (1.0 - (1.0 - k / E) ** batch) if batch > 1 else float(k)


def decode_bytes_per_step(p: dict, kv_len: float, batch: int = 1, touched: float = None) -> int:
    """SURVEY.md section 8(d): weights read once + KV rows of the visible window, bf16.  MoE: `touched` = measured number of
    distinct experts a layer streams per step (default: the expectation under uniform routing)."""
    dim, hd, hid, H, KV, V, L = p["dim"], p["head_dim"], p["hidden_dim"], p["n_heads"], p["n_kv_heads"], p["vocab_size"], p["n_layers"]
    p_attn = 2 * dim * H * hd + 2 * dim * KV * hd
    p_ffn = 3 * dim * hid
    moe = p.get("moe") or {}
    if moe:  # the router matrix + only the experts some token selected are read (moe.py:24-32)
        if touched is None:
            touched = experts_touched(moe["num_experts"], moe["num_experts_per_tok"], batch)
        p_ffn = touched * p_ffn + moe["num_experts"] * dim
    weights = 2 * (L * (p_attn + p_ffn + 2 * dim) + V * dim + dim)
    kv = 2 * L * batch * 2 * kv_len * KV * hd
    return int(weights + kv)


def prefill_flops(p: dict, T: int) -> float:
    dim, hd, hid, H, KV, V, L = p["dim"], p["head_dim"], p["hidden_dim"], p["n_heads"], p["n_kv_heads"], p["vocab_size"], p["n_layers"]
    p_attn = 2 * dim * H * hd + 2 * dim * KV * hd
    p_ffn = 3 * dim * hid
    moe = p.get("moe") or {}
    if moe:  # every token runs k experts + the router
        p_ffn = moe["num_experts_per_tok"] * p_ffn + moe["num_experts"] * dim
    W = p.get("sliding_window") or T
    vis = sum(min(i + 1, W) for i in range(T))
    return 2.0 * T * L * (p_attn + p_ffn) + 2.0 * T * V * dim + 4.0 * L * H * hd * vis


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def __enter__(self):
        exe = shutil.which("nvidia-smi")
        if exe:
            self.proc = subprocess.Popen([exe, f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50", "-i", str(self.index)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def wait_first(self, timeout_s: float = 3.0):
        """nvidia-smi needs a few hundred ms to start: without this a 60 ms timed region ends before the first sample."""
        t0 = time.perf_counter()
        while self.proc is not None and not self.rows and time.perf_counter() - t0 < timeout_s:
            time.sleep(0.02)
        self.rows.clear()  # samples from before the load started are not "under load"

    def __exit__(self, *exc):
        if self.proc:
            time.sleep(0.15)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        ok = [r for r in self.rows if len(r) >= 7 and r[0].replace(".", "").isdigit()]
        if not ok:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unparsable"]}
        reasons = []
        for i, name in enumerate(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]):
            if any(r[3 + i].lower().startswith("active") for r in ok):
                reasons.append(name)
        return {"sm_mhz": statistics.median(float(r[0]) for r in ok), "sm_max_mhz": float(ok[0][1]),
                "power_w_max": max(float(r[2]) for r in ok if r[2].replace(".", "").isdigit()), "samples": len(ok), "reasons": reasons}


def max_over_ranks(value: float, world: int, device) -> float:
    """Timing rule for N > 1: every rank times itself on the device, the job's time is the MAX over ranks."""
    if world <= 1:
        return float(value)
    t = torch.tensor([float(value)], device=device, dtype=torch.float64)
    torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
    return float(t.item())


def whole_job_tokens_per_s(replicas: int, batch: int, steps: int, elapsed_ms: float) -> float:
    return replicas * batch * steps * 1000.0 / elapsed_ms


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir: str, arrays: dict) -> None:
    """--dump-outputs: writes each tensor as out_dir/<name>.npy, floating point as float32 and token ids as float64 (exact), so
    that two builds run with the same arguments can be compared output for output.  A tensor larger than its share of
    DUMP_LIMIT_BYTES is replaced by a fixed seeded sample of its elements (flattened), written with their indices as
    <name>_index.npy."""
    import numpy as np

    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    share = DUMP_LIMIT_BYTES // len(arrays)
    for name, t in arrays.items():
        x = t.detach().cpu()
        x = (x.double() if not x.is_floating_point() else x.float()).numpy()
        if x.nbytes > share:  # a sampled element costs its own bytes + 8 for its index
            idx = np.sort(np.random.default_rng(0).choice(x.size, share // (x.itemsize + 8), replace=False))
            np.save(out / f"{name}_index.npy", idx.astype(np.float64))
            x = x.reshape(-1)[idx]
        np.save(out / f"{name}.npy", x)


# ------------------------------------------------------------------------------------------------ our arm
def build_gpu_model(p: dict, max_batch: int, seed: int = 0, expert_parallel=None):
    import mistral_inference_b200 as mi
    from mistral_inference_b200.transformer import Transformer

    args = mi.TransformerArgs.from_dict(dict(p))
    args.max_batch_size = max_batch
    dev = torch.device("cuda", torch.cuda.current_device())
    model = Transformer.empty(args, dev, torch.bfloat16, expert_parallel=expert_parallel)
    with torch.no_grad():
        for k, shp in synth.state_dict_shapes(p):  # stream tensor by tensor: no second copy of the checkpoint
            if model._owns_key(k):
                model._assign(k, synth.synth_tensor(k, shp, seed, torch.bfloat16, dev))
    return model.eval()


def moe_stats(model, batch: int):
    """(sum of distinct experts over MoE calls, calls) accumulated by moe_plan_kernel in the decode-sized row buffers."""
    ws = getattr(model, "_ws", None)
    tot = calls = 0
    for key, b in (ws._moe.items() if ws is not None else []):
        if key[0] == batch:
            h = b.plan[:8].tolist()
            tot, calls = tot + h[4], calls + h[5]
    return tot, calls


def timed_decode(model, cache, tok, steps: int, warmup: int, world: int, dev_index: int, sample_clocks: bool = True):
    """W warm-up + K timed decode steps with the token fed back on the device.  Returns (ms total max over ranks, us per launch
    of the hot-path launch (CUDA events on the launch stream, this rank), clocks summary, last token, fp32 logits [B, V] of the
    last step (the step's static buffer: valid until the next decode step))."""
    kern_ev = []
    last = {}

    def step(t, timed=False):
        if timed:
            a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a0.record()
            last["logits"] = model.decode_static(t, cache)
            a1.record()
            kern_ev.append((a0, a1))
        else:
            model.decode_static(t, cache)
        return model.last_argmax  # greedy pick made on the device (fused in the decode kernel / in the step's graph)

    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(dev_index) as clocks:  # started before the warm-up so that it is sampling when the (short) timed region runs
        if sample_clocks:
            clocks.wait_first()
        for _ in range(max(warmup, 3)):
            tok = step(tok)
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()
        e0.record()
        for _ in range(steps):
            tok = step(tok, timed=True)
        e1.record()
        torch.cuda.synchronize()
    ms = max_over_ranks(e0.elapsed_time(e1), world, torch.device("cuda", dev_index))
    kern_us = 1000.0 * sum(x.elapsed_time(y) for x, y in kern_ev) / len(kern_ev)
    return ms, kern_us, clocks.summary() if sample_clocks else None, tok, last["logits"]


def parity_check(model, p, prompt, seqlens, steps: int):
    """After the timed loop: the megakernel's greedy tokens over `steps` steps against the per-op kernel path (the path the
    oracle-checked op tests cover) teacher-forced on them, from identical prefilled caches.  Reported in the JSON line."""
    from mistral_inference_b200.cache import BufferCache

    L, B = p["n_layers"], len(seqlens)

    def prefilled():
        c = BufferCache(L, B, seqlens[0] + steps + 8, p["n_kv_heads"], p["head_dim"], p.get("sliding_window")).to(model.device, model.dtype)
        lg = model.forward(prompt, seqlens, c)
        return c, lg[torch.tensor(seqlens).cumsum(0) - 1].argmax(-1)

    cache, tok = prefilled()
    toks, mk_logits = [], []
    for _ in range(steps):
        toks.append(tok.clone())
        lg = model.decode_static(tok, cache)
        mk_logits.append(lg.clone())
        tok = model.last_argmax.clone()
    del cache
    os.environ["MB200_MEGAKERNEL"] = "0"
    os.environ["MB200_DECODE_GRAPH"] = "0"
    try:
        cache, _ = prefilled()
        match = decisive = decisive_match = 0
        worst = 0.0
        for s in range(steps):
            lg = model.forward(toks[s], [1] * B, cache)
            worst = max(worst, (lg - mk_logits[s]).abs().max().item())
            a, b = lg.argmax(-1), mk_logits[s].argmax(-1)
            top2 = lg.topk(2, dim=-1).values
            ulp = 2.0 ** (math.floor(math.log2(max(float(lg.abs().max()), 1e-30))) - 7)
            dec = (top2[:, 0] - top2[:, 1]) > 4 * ulp
            match += int((a == b).sum())
            decisive += int(dec.sum())
            decisive_match += int((a == b)[dec].sum())
    finally:
        os.environ.pop("MB200_MEGAKERNEL", None)
        os.environ.pop("MB200_DECODE_GRAPH", None)
    return {"steps": steps, "against": "per-op kernel path (oracle-checked op by op), teacher-forced on the megakernel's tokens, same prefilled cache",
            "token_match": f"{match}/{steps * B}", "decisive_picks": decisive, "decisive_match": decisive_match,
            "max_abs_logit_diff": round(worst, 5), "ok": decisive_match == decisive}


def run_ours(a, rank: int, world: int):
    import mistral_inference_b200 as mi  # noqa: F401
    from mistral_inference_b200 import _abi  # loads libmb200.so now: a missing build fails here, loudly
    from mistral_inference_b200.cache import BufferCache
    from mistral_inference_b200.generate import pick

    p = synth.shape(a.model)
    if a.layers:
        p["n_layers"] = a.layers
    L = p["n_layers"]
    dev_index = torch.cuda.current_device()
    expert = a.parallel == "expert" and world > 1
    model = build_gpu_model(p, a.batch, expert_parallel=(rank, world) if expert else None)
    replicas = 1 if expert else world
    max_seq = a.prefill + 2 * (a.steps + max(a.warmup, 32)) + 64
    W = p.get("sliding_window") or max_seq

    def fresh_cache():
        return BufferCache(L, a.batch, max_seq, p["n_kv_heads"], p["head_dim"], p.get("sliding_window")).to(model.device, model.dtype)

    # a different prompt per sequence (identical sequences would route identically: a batch of 8 would touch 2 experts, not ~7)
    prompt = torch.tensor(sum((synth.synth_prompt(a.prefill, p["vocab_size"], 7 + 13 * b) for b in range(a.batch)), []), device=model.device)
    seqlens = [a.prefill] * a.batch

    if os.environ.get("MB200_PROFILE") == "1":  # ncu --profile-from-start off: skip the synthetic-weight generation
        torch.cuda.profiler.start()
    # ---- prefill: median of 3 timed forwards after one untimed forward of the SAME length (first launches of a kernel variant
    # load its module).  For large batches the [T, V] logits do not fit (Nemo: 17 GB): time the hidden states + last-token head ----
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    full_logits = a.prefill * a.batch * p["vocab_size"] * 4 <= (4 << 30)
    times = []
    tok = None
    cache = None
    prefill_last = None
    for rep in range(4):
        del cache
        cache = fresh_cache()
        torch.cuda.synchronize()
        e0.record()
        if full_logits:
            logits = model.forward(prompt, seqlens, cache)
            last = logits[torch.tensor(seqlens).cumsum(0) - 1]
            del logits
        else:
            _, last = model.forward_logprobs(prompt, seqlens, cache, torch.full_like(prompt, -1))
        e1.record()
        torch.cuda.synchronize()
        if rep:
            times.append(e0.elapsed_time(e1))
        tok = last.argmax(-1)
        if a.dump_outputs and rep == 3:
            prefill_last = last.float().cpu()  # after the timed region: the copy is not timed
        del last
    prefill_ms = max_over_ranks(sorted(times)[1], world, model.device)
    pf = prefill_flops(p, a.prefill) * a.batch  # the lm head runs on every row in both variants (forward_logprobs: block by block)

    megakernel = model._megakernel_ok(a.batch)
    peaks = measured_peaks()
    n_gpus_bw = world if expert else 1

    # ---- e2e: the public API with HOST tokens: pinned H2D of the token, one decode step, D2H of (token, logprob) ----
    host_tok = torch.zeros(a.batch, dtype=torch.long).pin_memory()
    host_out = torch.zeros(a.batch, 2, dtype=torch.float32).pin_memory()
    dev_out = torch.zeros(a.batch, 2, dtype=torch.float32, device=model.device)
    nxt = torch.zeros(a.batch, dtype=torch.long, device=model.device)
    lp = torch.zeros(a.batch, dtype=torch.float32, device=model.device)
    host_tok.copy_(tok.cpu())

    def e2e_step():
        t = host_tok.to(model.device, non_blocking=True)
        lg = model.next_token_logits(t, cache)
        pick(lg, 0.0, 0.8, out=nxt, fused_argmax=model.last_argmax if model.last_argmax_valid_for(lg) else None)
        _abi.logprob_gather(lg, nxt, out=lp)
        dev_out[:, 0] = nxt
        dev_out[:, 1] = lp
        host_out.copy_(dev_out, non_blocking=True)
        torch.cuda.synchronize()
        host_tok[:] = host_out[:, 0].long()

    e2e_warmup = max(32, a.warmup)  # the first decode steps after the prefills of a fresh process run up to 5 % slow: settle first
    for _ in range(e2e_warmup):
        e2e_step()
    if world > 1:
        torch.distributed.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(a.steps):
        e2e_step()
    torch.cuda.synchronize()
    e2e_s = max_over_ranks(time.perf_counter() - t0, world, model.device)
    e2e_val = whole_job_tokens_per_s(replicas, a.batch, a.steps, e2e_s * 1000.0)
    tok = host_tok.to(model.device)

    # ---- decode: device-resident loop (value).  Runs after the end-to-end loop: the first decode steps right after the prefills of a
    # fresh process were measured up to 5 % slower than steady state on some boxes; W warm-up steps still precede the K timed ones ----
    st0 = moe_stats(model, a.batch)
    dec_ms, kern_us, clocks, tok, dec_logits = timed_decode(model, cache, tok, a.steps, a.warmup, world, dev_index)
    st1 = moe_stats(model, a.batch)
    if a.dump_outputs and rank == 0:
        dump_outputs(a.dump_outputs, {"decode_logits": dec_logits, "decode_next_token": tok, "prefill_last_logits": prefill_last})
    del dec_logits
    touched = (st1[0] - st0[0]) / (st1[1] - st0[1]) if st1[1] > st0[1] else None  # measured distinct experts per MoE layer call
    ms_per_step = dec_ms / a.steps
    value = whole_job_tokens_per_s(replicas, a.batch, a.steps, dec_ms)
    kv_len = min(W, a.prefill + e2e_warmup + a.steps + max(a.warmup, 3) + a.steps / 2.0)  # prefill + the e2e loop's steps + warm-up + half of the timed loop
    step_bytes = decode_bytes_per_step(p, kv_len, a.batch, touched)

    parity = None
    if rank == 0 and megakernel and not a.no_parity:
        parity = parity_check(model, p, prompt, seqlens, 64)
    del cache

    # ---- the sharded sub-record of an N > 1 replica line: expert-parallel Mixtral on the same GPUs ----
    sharded = None
    if world > 1 and not expert and not a.no_sharded:
        del model
        torch.cuda.empty_cache()
        try:
            sharded = run_sharded(a, rank, world, dev_index)
        except Exception as e:  # never lose the headline line to the sub-record
            sharded = {"error": f"{type(e).__name__}: {e}"[:300]}
        model = None

    # ---- roofline of the dominant kernel ----
    if rank != 0:
        return None
    traffic = None
    tf = REPO / "profiles" / "dominant_kernel_traffic.json"
    if tf.exists() and a.model == "mistral-7b" and not a.layers and a.batch == 1:  # the ncu capture is of exactly this workload
        traffic = json.loads(tf.read_text()).get("dram_bytes_per_launch")
    bw_peak = peaks["hbm_gbs"] * n_gpus_bw
    achieved = step_bytes / (kern_us * 1e-6) / 1e9
    if megakernel:
        kernel = f"decode_megakernel<{p['n_heads'] // p['n_kv_heads']}> (one persistent cooperative kernel per token: all layers + lm head + argmax)"
        timing = "CUDA events around every launch inside the timed decode loop (launch stream), mean of %d" % a.steps
    else:
        kernel = ("one CUDA-graph launch per step: decode_meta + per layer [rmsnorm, gemm_tcgen05<small batch> qkv+rope+ring write, attn_decode, "
                  "gemm wo+residual, rmsnorm, gemm gate/up+SiLU*mul | grouped MoE, gemm down+residual] + lm head + argmax_rows")
        timing = "CUDA events around every graph launch inside the timed decode loop, mean of %d" % a.steps
    roof = {"bound": "hbm", "kernel": kernel, "achieved": round(achieved, 1), "peak": bw_peak, "unit": "GB/s", "frac": round(achieved / bw_peak, 4),
            "traffic": traffic, "bytes_per_launch": step_bytes, "us_per_launch": round(kern_us, 2), "peak_source": peaks["source"], "timing": timing}
    if p.get("moe") and a.batch > 1:
        roof["distinct_experts_per_layer"] = round(touched, 3) if touched is not None else None
        roof["note"] = ("MoE bytes use the MEASURED number of distinct experts per layer and step (device-side counter of the routing plan)" if touched is not None
                        else "MoE bytes use the expected number of distinct experts per layer under uniform routing")

    cpu = cpu_baseline(a, p, bounded_seconds=20.0) if (world == 1 and not a.no_cpu_baseline) else None
    step_gbs = step_bytes / (ms_per_step * 1e-3) / 1e9
    prefill_kernels = ("gemm_tcgen05_kernel (tcgen05.mma/TMEM/TMA, 2-CTA clusters with multicast W tiles) + attn_prefill_tcgen05_kernel "
                       "(tcgen05 flash attention, S/P/O in TMEM) + rmsnorm/kv_ring_write" + (" + grouped expert GEMMs" if p.get("moe") else ""))
    per_layer = 9 if p.get("moe") else 7
    return {
        "metric": METRIC,
        "value": round(value, 2), "unit": "tokens/s", "n_gpus": world, "steps": a.steps, "warmup": max(a.warmup, 3),
        "ms_per_step": round(ms_per_step, 4), "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
        "data": f"synthetic (hash-seeded random-init weights of the {a.model} architecture, synthetic token ids)",
        "config": {"workload": f"{a.model} {L}L GQA {p['n_heads']}/{p['n_kv_heads']} sliding_window={p.get('sliding_window')} "
                               f"batch={a.batch} {a.prefill}-token prefill then decode at kv_len~{int(kv_len)}",
                   "parallelism": ("expert-sharded MoE over %d GPUs (experts e %% N == rank, rest replicated)" % world) if expert else
                                  ("replicas only" if world > 1 else "single GPU"),
                   "global_batch": a.batch * replicas, "seq_len": a.prefill,
                   "l2": f"inputs larger than L2 ({step_bytes / 1e9:.1f} GB streamed per step vs 126 MB L2)",
                   "decode_launch": "one persistent cooperative kernel per token (decode_megakernel)" if megakernel else "one CUDA-graph launch per step (device-side step state)",
                   "valid": a.layers in (None, 0)},
        "e2e": {"value": round(e2e_val, 2), "unit": "tokens/s", "h2d_bytes_per_step": 8 * a.batch, "d2h_bytes_per_step": 8 * a.batch,
                "warmup": e2e_warmup,
                "api": "Transformer.next_token_logits(pinned host token -> H2D, cache) + device pick + mb200_logprob_gather, (token, logprob) D2H, synchronised every step"},
        "gpu_launches": a.steps * (1 if megakernel else per_layer * L + 4),
        "clocks": clocks,
        "roofline": roof,
        "step_roofline": {"bound": "hbm", "algorithmic_bytes_per_step": step_bytes, "achieved": round(step_gbs, 1), "peak": bw_peak,
                          "unit": "GB/s", "frac": round(step_gbs / bw_peak, 4), "peak_source": peaks["source"]},
        "prefill": {"tokens": a.prefill * a.batch, "ms": round(prefill_ms, 2), "tflops": round(pf / prefill_ms / 1e9, 1),
                    "frac_of_burst_peak": round(pf / prefill_ms / 1e9 / (peaks["bf16_tflops"] * n_gpus_bw), 4), "algorithmic_flops": pf,
                    "lm_head": "all rows, [T, V] fp32 logits materialised" if full_logits else "all rows, block by block with the fused log-softmax + gather (the full [T, V] fp32 logits would not fit)",
                    "bound": "tensor", "peak_tflops": peaks["bf16_tflops"] * n_gpus_bw, "kernels": prefill_kernels},
        "parity": parity,
        "sharded": sharded,
        "cpu_baseline": cpu,
    }


def run_sharded(a, rank: int, world: int, dev_index: int):
    """Expert-parallel Mixtral decode on all `world` GPUs (SURVEY.md 8e; BASELINE configs[3]/[4]): 8x22B at 8 GPUs (B = 16),
    8x7B otherwise (B = 8).  value = B * K / max-over-ranks time; roofline against world x HBM bandwidth."""
    from mistral_inference_b200.cache import BufferCache

    name, B, P = ("mixtral-8x22b", 16, 512) if world >= 8 else ("mixtral-8x7b", 8, 512)
    p = synth.shape(name)
    if p["moe"]["num_experts"] % world:
        return {"skipped": f"{p['moe']['num_experts']} experts do not split over {world} ranks"}
    model = build_gpu_model(p, B, expert_parallel=(rank, world))
    K, Wm = min(a.steps, 32), max(a.warmup, 3)
    cache = BufferCache(p["n_layers"], B, P + 2 * (K + Wm) + 16, p["n_kv_heads"], p["head_dim"], None).to(model.device, model.dtype)
    prompt = torch.tensor(sum((synth.synth_prompt(P, p["vocab_size"], 11 + 13 * b) for b in range(B)), []), device=model.device)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for rep in range(2):  # the first forward loads modules and sets up the group's peer memory: time the second
        cache.reset()
        torch.cuda.synchronize()
        e0.record()
        _, last = model.forward_logprobs(prompt, [P] * B, cache, torch.full_like(prompt, -1))
        e1.record()
        torch.cuda.synchronize()
    prefill_ms = max_over_ranks(e0.elapsed_time(e1), world, model.device)
    tok = last.argmax(-1)
    st0 = moe_stats(model, B)
    ms, kern_us, _, _, _ = timed_decode(model, cache, tok, K, Wm, world, dev_index, sample_clocks=False)
    st1 = moe_stats(model, B)
    touched = (st1[0] - st0[0]) / (st1[1] - st0[1]) if st1[1] > st0[1] else None
    peaks = measured_peaks()
    step_bytes = decode_bytes_per_step(p, P + Wm + K / 2.0, B, touched)
    gbs = step_bytes / (ms / K * 1e-3) / 1e9
    moe = p["moe"]
    rows = B * moe["num_experts_per_tok"]
    comm = {"kind": "all-gather of the weighted expert output rows, written by the down-projection GEMM's epilogue straight into every rank's row "
                    "buffer (NVLink peer stores, CUDA-IPC mappings) + one flag handshake per MoE layer; no reduction, no NCCL call on the data path",
            "rows_per_layer": rows, "bytes_pushed_per_rank_per_layer": int(rows / world * (world - 1) * p["dim"] * 2), "moe_layers_per_step": p["n_layers"]}
    return {"workload": f"{name} expert-sharded over {world} GPUs, batch {B}, {P}-token prefill then decode", "tokens_per_s": round(B * K * 1000.0 / ms, 1),
            "ms_per_step": round(ms / K, 3), "steps": K, "prefill_ms": round(prefill_ms, 1), "algorithmic_bytes_per_step": step_bytes,
            "distinct_experts_per_layer": round(touched, 3) if touched is not None else None,
            "roofline": {"bound": "hbm", "achieved": round(gbs, 1), "peak": peaks["hbm_gbs"] * world, "unit": "GB/s", "frac": round(gbs / (peaks["hbm_gbs"] * world), 4)},
            "exchange": comm}


# ------------------------------------------------------------------------------------------------ CPU arm
def cpu_baseline(a, p: dict, bounded_seconds: float, steps: int = 0, full_depth: bool = False):
    """The reference's algorithm (oracle restatement: same torch CPU ops, same rounding points as mistral-inference's modules;
    the reference itself needs xformers + CUDA and cannot run) on the host cores, decode steps at the bench's context length.
    full_depth: every layer of the model (weights from torch's CPU generator -- timing depends on shapes only); otherwise a
    `n`-layer slice with a full kv ring + final norm + lm head, per-layer median x n_layers (labelled extrapolation)."""
    from oracle import restatement as R

    ncpu = os.cpu_count() or 1
    torch.set_num_threads(ncpu)
    moe = p.get("moe") or {}
    model_bytes = sum(math.prod(s) for _, s in synth.state_dict_shapes(p)) * 2
    try:
        avail = os.sysconf("SC_AVPHYS_PAGES") * os.sysconf("SC_PAGE_SIZE")
    except (ValueError, OSError):
        avail = 0
    full = full_depth and model_bytes * 1.25 < avail
    n = p["n_layers"] if full else min(p["n_layers"], 4)
    ps = dict(p, n_layers=n)
    oargs = R.OracleArgs(dim=p["dim"], n_layers=n, head_dim=p["head_dim"], hidden_dim=p["hidden_dim"], n_heads=p["n_heads"],
                         n_kv_heads=p["n_kv_heads"], norm_eps=p["norm_eps"], vocab_size=p["vocab_size"], max_batch_size=a.batch,
                         num_experts=moe.get("num_experts", 0), num_experts_per_tok=moe.get("num_experts_per_tok", 0),
                         sliding_window=p.get("sliding_window"))
    if full:
        g = torch.Generator().manual_seed(0)
        w = {}
        for k, shp in synth.state_dict_shapes(ps):
            bound = 0.25 if k.endswith("norm.weight") else float(shp[-1]) ** -0.5
            t = torch.empty(shp, dtype=torch.bfloat16)
            t.uniform_(-bound, bound, generator=g)
            w[k] = t + 1.0 if k.endswith("norm.weight") else t
    else:
        w = {k: synth.synth_tensor(k, shp, 0) for k, shp in synth.state_dict_shapes(ps)}
    om = R.OracleTransformer(oargs, w)
    W = p.get("sliding_window") or a.prefill
    cache = om.new_cache(a.prefill + 64)
    for l in range(n):  # synthetic ring contents: timing only depends on shapes
        cache.k[l].uniform_(-1, 1)
        cache.v[l].uniform_(-1, 1)
    cache.kv_seqlens = [a.prefill] * a.batch
    tok = torch.zeros(a.batch, dtype=torch.long)
    times = []
    t_all = time.perf_counter()
    with torch.inference_mode():
        # batch-1 bf16 matvecs do not scale to every core of a big host (128 threads measured 20x slower than 8): use the
        # thread count that is fastest for this workload (probed on two layers), and report it
        best = (None, float("inf"))
        probe = R.OracleTransformer(oargs, w, layer_ids=range(min(n, 2)))
        pc = probe.new_cache(a.prefill + 64)
        for nt in sorted({ncpu, min(ncpu, 64), min(ncpu, 32), min(ncpu, 16), min(ncpu, 8)}, reverse=True):
            torch.set_num_threads(nt)
            pc.kv_seqlens = [a.prefill] * a.batch
            probe.hidden(tok, [1] * a.batch, pc, last_stage=False)
            pc.kv_seqlens = [a.prefill] * a.batch
            t0 = time.perf_counter()
            probe.hidden(tok, [1] * a.batch, pc, last_stage=False)
            dt = time.perf_counter() - t0
            if dt < best[1]:
                best = (nt, dt)
        del pc, probe
        torch.set_num_threads(best[0])
        om.forward(tok, [1] * a.batch, cache)  # warm-up
        cache.kv_seqlens = [a.prefill] * a.batch
        while True:
            t0 = time.perf_counter()
            h = om.hidden(tok, [1] * a.batch, cache, last_stage=False)
            t1 = time.perf_counter()
            torch.nn.functional.linear(R.rms_norm(h, w["norm.weight"], p["norm_eps"]), w["output.weight"]).float()
            t2 = time.perf_counter()
            times.append((t1 - t0, t2 - t1))
            cache.kv_seqlens = [a.prefill] * a.batch  # stay at the same context length
            if (steps and len(times) >= steps) or (not steps and (time.perf_counter() - t_all > bounded_seconds or len(times) >= 50)):
                break
    t_layers = statistics.median(t[0] for t in times) / n
    t_head = statistics.median(t[1] for t in times)
    s_per_tok = t_layers * p["n_layers"] + t_head
    what = (f"{len(times)} decode steps of the FULL {p['n_layers']}-layer {a.model} (real shapes, kv ring at {W} positions), median step" if full else
            f"{len(times)} decode steps of a {n}-layer slice of {a.model} (real layer shapes, kv ring full at W={W}) + final norm + lm head, "
            f"per-layer median x {p['n_layers']} layers (labelled extrapolation: bounded sample)")
    return {"value": round(a.batch / s_per_tok, 4), "unit": "tokens/s", "cores": torch.get_num_threads(), "kind": "port",
            "host_cpus": ncpu, "full_depth": full, "sample": what, "ms_per_layer": round(t_layers * 1e3, 3), "ms_lm_head": round(t_head * 1e3, 3)}


def run_reference(a, rank: int, world: int):
    if rank != 0:
        return None
    p = synth.shape(a.model)
    if a.layers:
        p["n_layers"] = a.layers
    cpu = cpu_baseline(a, p, bounded_seconds=90.0, steps=max(a.steps, 1) + max(a.warmup, 0), full_depth=True)
    L = p["n_layers"]
    return {
        "impl": "reference", "metric": METRIC,
        "value": cpu["value"], "unit": "tokens/s", "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
        "ms_per_step": round(1000.0 * a.batch / cpu["value"], 2), "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
        "data": "synthetic",
        "config": {"workload": f"{a.model} {L}L GQA {p['n_heads']}/{p['n_kv_heads']} sliding_window={p.get('sliding_window')} "
                               f"batch={a.batch} decode at kv_len~{a.prefill}",
                   "arm": "the reference's algorithm on the host CPUs (oracle port with the reference's torch CPU ops and rounding points; the "
                          "reference itself needs xformers/CUDA and cannot run)", "full_depth": cpu["full_depth"]},
        "cpu_baseline": cpu,
        "e2e": {"value": cpu["value"], "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=128)
    ap.add_argument("--warmup", type=int, default=8)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--model", default="mistral-7b")
    ap.add_argument("--prefill", type=int, default=4096)
    ap.add_argument("--batch", type=int, default=1)
    ap.add_argument("--parallel", default="replicas", choices=["replicas", "expert"])
    ap.add_argument("--layers", type=int, default=0, help="debug only: fewer layers (marks the line invalid)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--no-sharded", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last timed decode step returned (fp32 "
                    "logits, greedy next token) and the last timed prefill's last-token logits as DIR/<name>.npy (at most 64 MB)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if a.impl == "reference":
        out = run_reference(a, rank, world)
    else:
        torch.cuda.set_device(local)
        if world > 1:
            torch.distributed.init_process_group("nccl", device_id=torch.device("cuda", local))
        out = run_ours(a, rank, world)
        if world > 1:
            torch.distributed.barrier()
            torch.distributed.destroy_process_group()
    if rank == 0 and out is not None:
        print(json.dumps(out))


if __name__ == "__main__":
    main()
