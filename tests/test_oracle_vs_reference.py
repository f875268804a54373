"""Pins the oracle restatement against the reference's own modules (run unmodified behind oracle/ref_shims.py).  What those
modules returned on each test's inputs is committed in tests/golden/reference_modules/ (oracle/make_golden.py --modules), so the
comparison runs without the reference: bit-exact on the fixture's torch build and CPU ISA, within the fp32-accumulation-order
tolerances of tests/test_oracle_golden.py on another CPU (which may pick other GEMM kernels)."""
import pytest
import torch

import synth
from oracle import restatement as R
from oracle.make_golden import (MODULES_DTYPES, MODULES_FILE, MODULES_GENERATE_CASES, ROPE_SAMPLE_ROWS, modules_generate_key,
                                tensor_sha256)

from .util import oracle_args, same_machine_as_golden


@pytest.fixture(scope="module")
def golden():
    import safetensors
    import safetensors.torch

    with safetensors.safe_open(str(MODULES_FILE), "pt") as f:
        meta = f.metadata()
    return safetensors.torch.load_file(str(MODULES_FILE)), meta


def _logit_tol(dtype) -> float:
    return 1e-4 if dtype == torch.float32 else 6e-2


@pytest.mark.parametrize("shape,over", MODULES_GENERATE_CASES)
@pytest.mark.parametrize("dtype", MODULES_DTYPES)
def test_generate_bit_exact(shape, over, dtype, golden):
    gold, meta = golden
    key = modules_generate_key(shape, over, dtype)
    counts = gold[key + "/logprob_counts"].tolist()
    t_ref = gold[key + "/tokens"].tolist()
    lp_ref = [x.tolist() for x in gold[key + "/logprobs"].split(counts)]
    p = synth.shape(shape, **over)
    om = R.OracleTransformer(oracle_args(p, 3), synth.synth_state_dict(p, 3, dtype))
    prompts = [synth.synth_prompt(n, p["vocab_size"], 40 + i) for i, n in enumerate([11, 9, 10])]
    t_or, lp_or = R.generate(prompts, om, max_tokens=9, chunk_size=4)
    assert t_ref == t_or
    if same_machine_as_golden(meta):
        assert lp_ref == lp_or  # python floats from identical fp32 tensors
    else:
        assert [len(x) for x in lp_or] == counts
        got = torch.tensor(sum(lp_or, []), dtype=torch.float64)
        torch.testing.assert_close(got, gold[key + "/logprobs"], rtol=0, atol=_logit_tol(dtype))


@pytest.mark.parametrize("dtype", MODULES_DTYPES)
def test_forward_without_cache_bit_exact(dtype, golden):
    """cache=None: unmasked, cross-sequence attention (SURVEY.md Appendix E-2)."""
    gold, meta = golden
    p = synth.shape("tiny")
    om = R.OracleTransformer(oracle_args(p, 2), synth.synth_state_dict(p, 3, dtype))
    toks = torch.tensor(synth.synth_prompt(13, p["vocab_size"], 5))
    with torch.inference_mode():
        b = om.forward(toks, [6, 7])
    a = gold[f"forward_no_cache/{str(dtype).removeprefix('torch.')}"]
    if same_machine_as_golden(meta):
        assert torch.equal(a, b)
    else:
        torch.testing.assert_close(b, a, rtol=0, atol=_logit_tol(dtype))


def test_elementwise_ops_bit_exact(golden):
    gold, meta = golden
    exact = same_machine_as_golden(meta)
    inp = {k.split("/")[-1]: v for k, v in gold.items() if k.startswith("elementwise/in/")}

    def check(got, want):
        if exact:
            assert torch.equal(got, want)
        else:
            torch.testing.assert_close(got, want)

    check(R.rms_norm(inp["x"], inp["w"], 1e-5), gold["elementwise/rms_norm"])
    table = R.rope_table(128, 1000, 1e6)
    if exact:
        assert tensor_sha256(torch.view_as_real(table)) == meta["rope_table_sha256"]
    check(torch.view_as_real(table)[ROPE_SAMPLE_ROWS], gold["elementwise/rope_table_rows"])
    fc = table[inp["positions"]]
    for got, name in zip(R.apply_rope(inp["q"], inp["k"], fc), ("rope_q", "rope_k")):
        check(got, gold[f"elementwise/{name}"])
