"""Import shims that let the UNMODIFIED reference modules run on CPU in this container
(TEST INFRASTRUCTURE -- see oracle/__init__.py).

The reference (`/root/reference/src/mistral_inference`) imports two packages that are not
installed and cannot be installed (no network): `xformers` (transformer_layers.py:6-7,
cache.py:5-10, vision_encoder.py) and `simple_parsing` (args.py:4, moe.py:6, lora.py:9).
`install()` registers minimal stand-ins in `sys.modules` and puts the reference's `src/` on
`sys.path`; after that `import mistral_inference.transformer` etc. work unmodified.

Only usable where a checkout of the reference is installed (MISTRAL_REFERENCE_SRC): used by
`oracle/make_golden.py` to produce tests/golden/, the fixtures that pin the restatement.  Mask
semantics: SURVEY.md Appendix B.
"""
import dataclasses
import os
import sys
import types
import typing
from typing import Any, List, Optional, Sequence

import torch

from .attention_ref import attend_block, local_causal_allowed

REFERENCE_SRC = os.environ.get("MISTRAL_REFERENCE_SRC", "/root/reference/src")


def reference_available() -> bool:
    return os.path.isdir(os.path.join(REFERENCE_SRC, "mistral_inference"))


# ----------------------------------------------------------------------------- simple_parsing
class Serializable:
    """Stand-in for simple_parsing.helpers.Serializable: only `from_dict` is used
    (transformer.py:306-307).  Recurses into dataclass-typed fields (moe / lora / vision_encoder)."""

    @classmethod
    def from_dict(cls, d: dict, drop_extra_fields: Any = None):  # noqa: ARG003
        hints = typing.get_type_hints(cls)
        kwargs = {}
        for f in dataclasses.fields(cls):
            if f.name not in d:
                continue
            val = d[f.name]
            tp = hints.get(f.name)
            sub = _dataclass_in(tp)
            if isinstance(val, dict) and sub is not None:
                val = sub.from_dict(val) if hasattr(sub, "from_dict") else sub(**val)
            kwargs[f.name] = val
        return cls(**kwargs)


def _dataclass_in(tp):
    if tp is None:
        return None
    if dataclasses.is_dataclass(tp):
        return tp
    for a in typing.get_args(tp):
        r = _dataclass_in(a)
        if r is not None:
            return r
    return None


# ----------------------------------------------------------------------------- xformers masks
class AttentionBias:
    pass


class BlockDiagonalMask(AttentionBias):
    """Block-diagonal over sequences; optional causal / local-window refinements."""

    def __init__(self, q_seqlen: Sequence[int], kv_seqlen: Sequence[int], causal: bool = False,
                 window: Optional[int] = None, from_bottomright: bool = False):
        assert len(q_seqlen) == len(kv_seqlen)
        self.q_seqlen = list(q_seqlen)
        self.kv_seqlen = list(kv_seqlen)
        self.causal = causal
        self.window = window
        self.from_bottomright = from_bottomright

    @classmethod
    def from_seqlens(cls, q_seqlen: Sequence[int], kv_seqlen: Optional[Sequence[int]] = None):
        return cls(q_seqlen, q_seqlen if kv_seqlen is None else kv_seqlen)

    def make_local_attention_from_bottomright(self, window_size: int):
        return BlockDiagonalMask(self.q_seqlen, self.kv_seqlen, causal=True, window=window_size, from_bottomright=True)

    def block_allowed(self, b: int, device=None) -> Optional[torch.Tensor]:
        s, n = self.q_seqlen[b], self.kv_seqlen[b]
        if not self.causal:
            return None
        return local_causal_allowed(s, n, self.window, device)


class BlockDiagonalCausalMask(BlockDiagonalMask):
    def __init__(self, q_seqlen, kv_seqlen, window: Optional[int] = None):
        super().__init__(q_seqlen, kv_seqlen, causal=True, window=window)

    @classmethod
    def from_seqlens(cls, q_seqlen: Sequence[int], kv_seqlen: Optional[Sequence[int]] = None):
        return cls(q_seqlen, q_seqlen if kv_seqlen is None else kv_seqlen)

    def make_local_attention(self, window_size: int):
        return BlockDiagonalCausalMask(self.q_seqlen, self.kv_seqlen, window=window_size)


class BlockDiagonalCausalWithOffsetPaddedKeysMask(AttentionBias):
    """Sequence b's keys live in the padded block [b*pad, b*pad+pad); only the first
    kv_seqlen[b] are valid; causal aligned bottom-right."""

    def __init__(self, q_seqlen, kv_padding: int, kv_seqlen):
        self.q_seqlen = list(q_seqlen)
        self.kv_padding = kv_padding
        self.kv_seqlen = list(kv_seqlen)

    @classmethod
    def from_seqlens(cls, q_seqlen: Sequence[int], kv_padding: int, kv_seqlen: Sequence[int]):
        assert all(k <= kv_padding for k in kv_seqlen)
        return cls(q_seqlen, kv_padding, kv_seqlen)


def memory_efficient_attention(query: torch.Tensor, key: torch.Tensor, value: torch.Tensor,
                               attn_bias: Optional[AttentionBias] = None, **_: Any) -> torch.Tensor:
    """[1, S, H, hd] in, contiguous [1, Sq, H, hd] out (the reference `.view`s it,
    transformer_layers.py:89)."""
    assert query.shape[0] == 1 and key.shape[0] == 1 and value.shape[0] == 1
    q, k, v = query[0], key[0], value[0]
    if attn_bias is None:
        return attend_block(q, k, v, None)[None]
    outs: List[torch.Tensor] = []
    if isinstance(attn_bias, BlockDiagonalCausalWithOffsetPaddedKeysMask):
        qo = 0
        for b, (s, n) in enumerate(zip(attn_bias.q_seqlen, attn_bias.kv_seqlen)):
            k0 = b * attn_bias.kv_padding
            allowed = local_causal_allowed(s, n, None, q.device)
            outs.append(attend_block(q[qo:qo + s], k[k0:k0 + n], v[k0:k0 + n], allowed))
            qo += s
        assert qo == q.shape[0]
    elif isinstance(attn_bias, BlockDiagonalMask):
        qo = ko = 0
        for b, (s, n) in enumerate(zip(attn_bias.q_seqlen, attn_bias.kv_seqlen)):
            outs.append(attend_block(q[qo:qo + s], k[ko:ko + n], v[ko:ko + n], attn_bias.block_allowed(b, q.device)))
            qo += s
            ko += n
        assert qo == q.shape[0] and ko == k.shape[0], (qo, q.shape, ko, k.shape)
    else:
        raise TypeError(f"unsupported attn_bias {type(attn_bias)}")
    return torch.cat(outs, dim=0)[None].contiguous()


# ----------------------------------------------------------------------------- install
_installed = False


def install() -> None:
    """Idempotent.  Raises if the reference tree is absent."""
    global _installed
    if _installed:
        return
    if not reference_available():
        raise RuntimeError(f"reference source tree not found at {REFERENCE_SRC}")

    sp = types.ModuleType("simple_parsing")
    sph = types.ModuleType("simple_parsing.helpers")
    sph.Serializable = Serializable
    sp.helpers = sph
    sys.modules.setdefault("simple_parsing", sp)
    sys.modules.setdefault("simple_parsing.helpers", sph)

    xf = types.ModuleType("xformers")
    xo = types.ModuleType("xformers.ops")
    xfm = types.ModuleType("xformers.ops.fmha")
    xab = types.ModuleType("xformers.ops.fmha.attn_bias")
    for cls in (AttentionBias, BlockDiagonalMask, BlockDiagonalCausalMask, BlockDiagonalCausalWithOffsetPaddedKeysMask):
        setattr(xab, cls.__name__, cls)
    xfm.memory_efficient_attention = memory_efficient_attention
    xfm.attn_bias = xab
    xo.fmha = xfm
    xo.memory_efficient_attention = memory_efficient_attention
    xf.ops = xo
    sys.modules.setdefault("xformers", xf)
    sys.modules.setdefault("xformers.ops", xo)
    sys.modules.setdefault("xformers.ops.fmha", xfm)
    sys.modules.setdefault("xformers.ops.fmha.attn_bias", xab)

    if REFERENCE_SRC not in sys.path:
        sys.path.insert(0, REFERENCE_SRC)
    _installed = True


def import_reference():
    """Returns the reference's (transformer, generate, cache, args) modules."""
    install()
    import mistral_inference.args as r_args  # type: ignore
    import mistral_inference.cache as r_cache  # type: ignore
    import mistral_inference.generate as r_generate  # type: ignore
    import mistral_inference.transformer as r_transformer  # type: ignore

    return types.SimpleNamespace(transformer=r_transformer, generate=r_generate, cache=r_cache, args=r_args)
