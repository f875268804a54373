"""bench.py's roofline numerators against an independent count made from the checkpoint's own tensor shapes (SURVEY.md 8(d)):
algorithmic bytes of one batch-1 decode step = every weight byte the step must read once + the visible KV rows."""
import math

import bench
import synth


def _weight_bytes_from_shapes(p: dict) -> int:
    moe = p.get("moe") or {}
    total = 0
    for key, shape in synth.state_dict_shapes(p):
        if key == "tok_embeddings.weight":
            continue  # one row gathered per token: noise
        n = math.prod(shape) * 2
        if moe and ".experts." in key:
            total += n * moe["num_experts_per_tok"] / moe["num_experts"]  # k of E experts are streamed at batch 1
        else:
            total += n
    return int(total)


def test_decode_bytes_dense_and_moe():
    for name in ("mistral-7b", "mixtral-8x7b", "tiny", "tiny-moe"):
        p = synth.shape(name)
        kv_len = 4096
        kv = 2 * p["n_layers"] * 2 * kv_len * p["n_kv_heads"] * p["head_dim"]
        assert bench.decode_bytes_per_step(p, kv_len) == _weight_bytes_from_shapes(p) + kv, name
    assert bench.decode_bytes_per_step(synth.shape("mistral-7b"), 4096) == 14_758_191_104  # the bench line's bytes_per_launch


def test_dump_outputs_dtypes_and_size_cap(tmp_path):
    """--dump-outputs: float32 logits and float64 token ids as <name>.npy; a tensor over its share of the 64 MB cap is replaced by
    the same seeded sample on every run, with its indices."""
    import numpy as np
    import torch

    big = torch.arange(3 * (1 << 22), dtype=torch.float32).view(3, -1)  # 48 MB: over a third of 64 MB
    arrays = {"logits": torch.ones(2, 5, dtype=torch.bfloat16), "token": torch.tensor([7, 2**40 + 1]), "big": big}
    for d in (tmp_path / "a", tmp_path / "b"):
        bench.dump_outputs(str(d), arrays)
    assert sorted(p.name for p in (tmp_path / "a").iterdir()) == ["big.npy", "big_index.npy", "logits.npy", "token.npy"]
    lg, tk = np.load(tmp_path / "a" / "logits.npy"), np.load(tmp_path / "a" / "token.npy")
    assert lg.dtype == np.float32 and lg.shape == (2, 5) and (lg == 1).all()
    assert tk.dtype == np.float64 and tk.tolist() == [7, 2**40 + 1]
    assert sum(p.stat().st_size for p in (tmp_path / "a").iterdir()) <= bench.DUMP_LIMIT_BYTES
    x, idx = np.load(tmp_path / "a" / "big.npy"), np.load(tmp_path / "a" / "big_index.npy")
    assert np.array_equal(x, big.numpy().reshape(-1)[idx.astype(np.int64)])
    assert np.array_equal(x, np.load(tmp_path / "b" / "big.npy"))


def test_prefill_flops_counts_every_linear_and_the_causal_half():
    p, T = synth.shape("mistral-7b"), 4096
    linear_params = sum(math.prod(s) for k, s in synth.state_dict_shapes(p) if len(s) == 2 and k != "tok_embeddings.weight")
    attn = 4.0 * p["n_layers"] * p["n_heads"] * p["head_dim"] * (T * (T + 1) // 2)  # QK^T and PV over the visible keys
    assert bench.prefill_flops(p, T) == 2.0 * T * linear_params + attn
