"""Generate tests/golden/*.safetensors from the UNMODIFIED reference modules
(TEST INFRASTRUCTURE -- see oracle/__init__.py).

Run where a checkout of the reference is installed (MISTRAL_REFERENCE_SRC = its src/ directory):
    python -m oracle.make_golden [--config1 | --modules | --all]
The tests must not need the reference, so its outputs on small seeded cases are committed as
fixtures.  Each fixture holds the outputs of the reference's own `Transformer.forward` /
`generate` (mistral_inference/transformer.py:221-242, generate.py:43-148) imported behind
oracle/ref_shims.py, on weights from synth (bit-reproducible anywhere).

Cases follow SURVEY.md section 8c "tests to carry over": ragged batch greedy decode; ring that
wraps (sliding_window < length); list-valued sliding_window; 8-expert top-2 MoE;
max_batch_size > B; chunked re-prefill (the reference's own consistency property).
"""
import json
import sys
from pathlib import Path
from typing import Dict, List

import torch

REPO = Path(__file__).resolve().parents[1]
if str(REPO) not in sys.path:
    sys.path.insert(0, str(REPO))

import synth  # noqa: E402
from oracle import ref_shims  # noqa: E402

GOLDEN_DIR = REPO / "tests" / "golden"

# name -> (shape name, param overrides, dtype, prompts (lengths), max_tokens, max_batch_size, chunk_size for re-prefill)
CASES: Dict[str, dict] = {
    "dense_full": dict(shape="tiny", over={}, dtype="bfloat16", prompt_lens=[8, 4, 4, 4], max_tokens=7, max_batch=4, chunk=None),
    "dense_w4_chunk5": dict(shape="tiny", over={"sliding_window": 4}, dtype="bfloat16", prompt_lens=[8, 10], max_tokens=8,
                            max_batch=3, chunk=5),
    "dense_wlist": dict(shape="tiny", over={"sliding_window": [3, None]}, dtype="bfloat16", prompt_lens=[8, 10], max_tokens=8,
                        max_batch=2, chunk=5),
    "moe_full": dict(shape="tiny-moe", over={}, dtype="bfloat16", prompt_lens=[9, 7, 8], max_tokens=6, max_batch=3, chunk=4),
    "moe_w4": dict(shape="tiny-moe", over={"sliding_window": 4}, dtype="bfloat16", prompt_lens=[9, 7], max_tokens=6, max_batch=2,
                   chunk=4),
    "dense_full_fp32": dict(shape="tiny", over={}, dtype="float32", prompt_lens=[8, 4, 4, 4], max_tokens=7, max_batch=4, chunk=None),
}


def case_inputs(case: dict, seed: int):
    p = synth.shape(case["shape"], **case["over"])
    prompts = [synth.synth_prompt(n, p["vocab_size"], seed * 100 + i) for i, n in enumerate(case["prompt_lens"])]
    return p, prompts


def run_reference(case: dict, seed: int = 1) -> Dict[str, torch.Tensor]:
    ref = ref_shims.import_reference()
    p, prompts = case_inputs(case, seed)
    dtype = getattr(torch, case["dtype"])
    args = ref.args.TransformerArgs.from_dict(dict(p))
    args.max_batch_size = case["max_batch"]
    with torch.device("meta"):
        model = ref.transformer.Transformer(args)
    model.load_state_dict(synth.synth_state_dict(p, seed, dtype), assign=True, strict=True)
    model = model.to(device="cpu", dtype=dtype).eval()

    recorded: List[torch.Tensor] = []
    orig_forward = model.forward

    def recording_forward(*a, **kw):
        out = orig_forward(*a, **kw)
        recorded.append(out.clone())
        return out

    model.forward = recording_forward  # instance attribute; the reference code itself is untouched
    toks, logprobs = ref.generate.generate(prompts, model, max_tokens=case["max_tokens"], temperature=0.0)
    out: Dict[str, torch.Tensor] = {}
    out["prefill_logits"] = recorded[0]  # [sum(prompt_lens), V] fp32
    out["decode_logits"] = torch.stack(recorded[1:], 0)  # [max_tokens, B, V] fp32 (last one is never sampled)
    out["tokens"] = torch.tensor(toks, dtype=torch.int64)
    out["logprobs"] = torch.tensor(sum(logprobs, []), dtype=torch.float64)
    # the reference's own consistency check: re-prefill prompt+generated (optionally chunked), max_tokens=0
    recorded.clear()
    full = [pr + t for pr, t in zip(prompts, toks)]
    gen2, logprobs2 = ref.generate.generate(full, model, max_tokens=0, temperature=0.0, chunk_size=case["chunk"])
    assert gen2 == []
    out["reprefill_logprobs"] = torch.tensor(sum(logprobs2, []), dtype=torch.float64)
    out["reprefill_logits"] = torch.cat(recorded, 0)  # chunks concatenated in call order
    return out


# ---- BASELINE.json configs[0]: "Mistral-7B shape, random-init bf16, 1 layer, batch=1, 128-token prompt + 32 decode on CPU
# (reference path, plumbing)".  The full logits would be 21 MB; the fixture keeps what pins the path: the greedy tokens, every
# log-probability generate() returns, the top-64 (value, index) of each step's logits and the first 256 vocabulary columns of
# the prompt's logits.  With random-init weights the two largest of 32000 bf16 logits are a few ulps apart on average (the gap
# of the top two order statistics is ~8 ulps, exponentially distributed), so over 32 steps some pick is always a near-tie that
# any two correct implementations may resolve differently.  The fixture therefore records the reference's top-1/top-2 margin of
# every step (in bf16 ulps); a step is DECISIVE when the margin is >= 3 ulps.  Token ids must be identical at every decisive
# step (teacher-forced), and the free-running generate() must reproduce the reference's ids up to the first non-decisive step.
# Among the first few weight seeds the one with the longest decisive prefix is kept.
CONFIG1 = dict(shape="mistral-7b", over={"n_layers": 1}, dtype="bfloat16", prompt_lens=[128], max_tokens=32, max_batch=1, chunk=None)
MIN_MARGIN_ULPS = 3
TOPK = 64


def bf16_ulp(x: torch.Tensor) -> torch.Tensor:
    """Spacing of bf16 numbers at |x| (8 significand bits)."""
    return torch.pow(2.0, torch.floor(torch.log2(x.abs().clamp_min(1e-30))) - 7)


def run_config1(max_seeds: int = 6):
    ref = ref_shims.import_reference()
    case = CONFIG1
    dtype = torch.bfloat16
    best = None
    for seed in range(1, max_seeds + 1):
        p, prompts = case_inputs(case, seed)
        args = ref.args.TransformerArgs.from_dict(dict(p))
        args.max_batch_size = case["max_batch"]
        with torch.device("meta"):
            model = ref.transformer.Transformer(args)
        model.load_state_dict(synth.synth_state_dict(p, seed, dtype), assign=True, strict=True)
        model = model.to(device="cpu", dtype=dtype).eval()
        recorded: List[torch.Tensor] = []
        orig_forward = model.forward

        def recording_forward(*a, **kw):
            out = orig_forward(*a, **kw)
            recorded.append(out.clone())
            return out

        model.forward = recording_forward
        toks, logprobs = ref.generate.generate(prompts, model, max_tokens=case["max_tokens"], temperature=0.0)
        # logits each of the 32 picks was made from: last prefill row, then the decode steps (the final forward is never sampled)
        picked_from = torch.cat([recorded[0][-1:]] + [r for r in recorded[1:-1]], 0)  # [32, V]
        top = picked_from.topk(TOPK, dim=-1)
        margins = (top.values[:, 0] - top.values[:, 1]) / bf16_ulp(top.values[:, 0])
        weak = (margins < MIN_MARGIN_ULPS).nonzero().flatten().tolist()
        prefix = weak[0] if weak else case["max_tokens"]
        print(f"config1 seed {seed}: decisive prefix {prefix}/32 steps, {32 - len(weak)} decisive steps, min margin {margins.min().item():.1f} ulps", flush=True)
        if best is None or prefix > best[0]:
            out = {"tokens": torch.tensor(toks, dtype=torch.int64), "logprobs": torch.tensor(sum(logprobs, []), dtype=torch.float64),
                   "topk_values": top.values.contiguous(), "topk_indices": top.indices.contiguous(), "margin_ulps": margins.contiguous(),
                   "prefill_logits_head": recorded[0][:, :256].contiguous()}  # first 256 vocab columns of all 128 prompt rows
            best = (prefix, seed, out)
        del model
        if prefix == case["max_tokens"]:
            break
    return best[1], best[0], best[2]


# ---- tests/test_oracle_vs_reference.py: what the reference's modules return on the inputs of each of its tests, so the restatement
# is pinned against the reference anywhere, not only where the reference tree is installed.  The rope table (1000 x 64 complex) is
# stored as the SHA-256 of its bytes plus a sample of rows; everything else is stored whole (about 100 KB in all).
MODULES_FILE = GOLDEN_DIR / "reference_modules" / "outputs.safetensors"
MODULES_GENERATE_CASES = [("tiny", {}), ("tiny", {"sliding_window": 5}), ("tiny", {"sliding_window": [4, None]}),
                          ("tiny-moe", {}), ("tiny-moe", {"sliding_window": 3})]
MODULES_DTYPES = [torch.bfloat16, torch.float32]
ROPE_SAMPLE_ROWS = sorted(set(range(0, 1000, 25)) | {1, 2, 500, 501, 998, 999})


def modules_generate_key(shape: str, over: dict, dtype: torch.dtype) -> str:
    return f"generate/{shape}/{json.dumps(over, sort_keys=True)}/{str(dtype).removeprefix('torch.')}"


def elementwise_inputs():
    """The inputs of the element-wise comparison (seeded torch CPU generator; stored with the outputs)."""
    torch.manual_seed(0)
    x = torch.randn(7, 256).to(torch.bfloat16)
    w = (1 + 0.1 * torch.randn(256)).to(torch.bfloat16)
    q = torch.randn(7, 4, 128).to(torch.bfloat16)
    k = torch.randn(7, 2, 128).to(torch.bfloat16)
    return {"x": x, "w": w, "q": q, "k": k, "positions": torch.tensor([0, 1, 2, 500, 501, 998, 999])}


def tensor_sha256(t: torch.Tensor) -> str:
    import hashlib

    return hashlib.sha256(t.contiguous().view(torch.uint8).numpy().tobytes()).hexdigest()


def _ref_model(ref, p: dict, max_batch: int, dtype: torch.dtype, seed: int = 3):
    args = ref.args.TransformerArgs.from_dict(dict(p))
    args.max_batch_size = max_batch
    with torch.device("meta"):
        m = ref.transformer.Transformer(args)
    m.load_state_dict(synth.synth_state_dict(p, seed, dtype), assign=True, strict=True)
    return m.eval()


def run_modules():
    ref = ref_shims.import_reference()
    import mistral_inference.rope as r_rope  # type: ignore
    import mistral_inference.transformer_layers as r_layers  # type: ignore

    out: Dict[str, torch.Tensor] = {}
    for shape, over in MODULES_GENERATE_CASES:
        for dtype in MODULES_DTYPES:
            p = synth.shape(shape, **over)
            rm = _ref_model(ref, p, 3, dtype)
            prompts = [synth.synth_prompt(n, p["vocab_size"], 40 + i) for i, n in enumerate([11, 9, 10])]
            toks, logprobs = ref.generate.generate(prompts, rm, max_tokens=9, temperature=0.0, chunk_size=4)
            key = modules_generate_key(shape, over, dtype)
            out[key + "/tokens"] = torch.tensor(toks, dtype=torch.int64)
            out[key + "/logprobs"] = torch.tensor(sum(logprobs, []), dtype=torch.float64)  # python floats of fp32 values: exact
            out[key + "/logprob_counts"] = torch.tensor([len(x) for x in logprobs], dtype=torch.int64)
    for dtype in MODULES_DTYPES:
        p = synth.shape("tiny")
        rm = _ref_model(ref, p, 2, dtype)
        toks = torch.tensor(synth.synth_prompt(13, p["vocab_size"], 5))
        with torch.inference_mode():
            out[f"forward_no_cache/{str(dtype).removeprefix('torch.')}"] = rm.forward(toks, seqlens=[6, 7]).contiguous()

    inp = elementwise_inputs()
    out.update({f"elementwise/in/{k}": v for k, v in inp.items()})
    norm = r_layers.RMSNorm(256, eps=1e-5)
    norm.weight.data = inp["w"]
    with torch.no_grad():
        out["elementwise/rms_norm"] = norm(inp["x"]).contiguous()
    table = r_rope.precompute_freqs_cis(128, 1000, 1e6)
    out["elementwise/rope_table_rows"] = torch.view_as_real(table)[ROPE_SAMPLE_ROWS].contiguous()
    xq, xk = r_rope.apply_rotary_emb(inp["q"], inp["k"], table[inp["positions"]])
    out["elementwise/rope_q"], out["elementwise/rope_k"] = xq.contiguous(), xk.contiguous()
    meta = {"torch": torch.__version__, "cpu_capability": torch.backends.cpu.get_cpu_capability(),
            "rope_table_sha256": tensor_sha256(torch.view_as_real(table)),
            "reference": "mistralai/mistral-inference@2557e12 (v1.6.0) modules, unmodified, via oracle/ref_shims.py"}
    return out, meta


def main() -> None:
    GOLDEN_DIR.mkdir(parents=True, exist_ok=True)
    import safetensors.torch

    if "--config1" in sys.argv or "--all" in sys.argv:
        seed, prefix, out = run_config1()
        meta = {"case": json.dumps(CONFIG1), "seed": str(seed), "decisive_prefix": str(prefix), "min_margin_ulps": str(MIN_MARGIN_ULPS), "torch": torch.__version__,
                "cpu_capability": torch.backends.cpu.get_cpu_capability(),
                "reference": "mistralai/mistral-inference@2557e12 (v1.6.0) modules, unmodified, via oracle/ref_shims.py"}
        safetensors.torch.save_file(out, str(GOLDEN_DIR / "config1_7b_1layer.safetensors"), metadata=meta)
        print(f"config1_7b_1layer: seed={seed} tokens={out['tokens'].tolist()}")
        if "--config1" in sys.argv:
            return

    if "--modules" in sys.argv or "--all" in sys.argv:
        out, meta = run_modules()
        MODULES_FILE.parent.mkdir(parents=True, exist_ok=True)
        safetensors.torch.save_file(out, str(MODULES_FILE), metadata=meta)
        print(f"{MODULES_FILE.relative_to(REPO)}: {len(out)} tensors, {sum(v.numel() * v.element_size() for v in out.values())} bytes")
        if "--modules" in sys.argv:
            return

    for name, case in CASES.items():
        out = run_reference(case)
        # the reference's property, on the reference itself (fp32 bound of tests/test_generate.py:63 is 5e-4; bf16 is looser)
        n = min(len(out["logprobs"]), len(out["reprefill_logprobs"]))
        meta = {
            "case": json.dumps(case),
            "seed": "1",
            "torch": torch.__version__,
            "cpu_capability": torch.backends.cpu.get_cpu_capability(),
            "reference": "mistralai/mistral-inference@2557e12 (v1.6.0) modules, unmodified, via oracle/ref_shims.py",
        }
        safetensors.torch.save_file({k: v.contiguous() for k, v in out.items()}, str(GOLDEN_DIR / f"{name}.safetensors"), metadata=meta)
        print(f"{name}: tokens={out['tokens'].tolist()} prefill_logits={tuple(out['prefill_logits'].shape)} "
              f"bytes={sum(v.numel() * v.element_size() for v in out.values())} n_logprobs={n}")


if __name__ == "__main__":
    main()
