"""TEST INFRASTRUCTURE (build container only): runs the UNMODIFIED reference implementation from
/root/reference so the oracle restatement can be pinned against it and golden fixtures generated.

/root/reference does not exist on the GPU box, so nothing that runs there imports this module
(tests guard it with ``reference_available()``).

Two shims are needed to execute the reference offline (SURVEY.md appendix A):
  * ``Tokenizer.from_pretrained`` (moondream/torch/moondream.py:89) needs the network -> stub whose
    ``decode`` prints the ids, so generated token ids can be read back from the text API;
  * weights: seeded synthetic tensors in the canonical state_dict layout (moondream_b200.synth).
"""
from __future__ import annotations

import os
import sys
from typing import Dict, List

import torch

REFERENCE_ROOT = "/root/reference"


def reference_available() -> bool:
    return os.path.isdir(os.path.join(REFERENCE_ROOT, "moondream", "torch"))


class _Enc:
    def __init__(self, ids):
        self.ids = ids


class StubTokenizer:
    """`encode` maps whitespace-separated integers to ids (anything else hashes into the vocab);
    `decode` prints ids space-separated so the streamed text is a lossless dump of the tokens."""

    def __init__(self, vocab_size: int):
        self.vocab_size = vocab_size

    def encode(self, text: str):
        ids = []
        for tok in text.split():
            try:
                ids.append(int(tok) % self.vocab_size)
            except ValueError:
                ids.append(10 + (sum(tok.encode()) * 2654435761 % (self.vocab_size - 10)))
        return _Enc(ids)

    def decode(self, ids: List[int]) -> str:
        return "".join(f"{int(i)} " for i in ids)


class PieceTokenizer:
    """A tokenizer whose pieces exercise every flush rule of the reference's streaming detokeniser
    (moondream.py:476-537): words with leading spaces, bare suffixes, newlines, CJK characters, punctuation."""

    PIECES = [" the", " cat", "s", " sat", "\n", "\u6f22", "\u5b57", " on", ",", " a", " mat", ".", "\n\n",
              " \u65e5\u672c", "\u00e9", " ", "ing", " x\n", "\u3400", " end"]

    def __init__(self, pieces=None):
        self.pieces = list(pieces) if pieces is not None else list(self.PIECES)

    def encode(self, text: str):
        return _Enc([sum(text.encode()) % len(self.pieces)])

    def decode(self, ids: List[int]) -> str:
        return "".join(self.pieces[int(i) % len(self.pieces)] for i in ids)


def load_reference_model(cfg, state_dict: Dict[str, torch.Tensor]):
    """Construct the reference MoondreamModel (CPU, bf16) with `state_dict` loaded."""
    if not reference_available():
        raise RuntimeError("/root/reference is not present on this box")
    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)
    import moondream.torch.moondream as ref_md
    from moondream.torch.config import MoondreamConfig as RefConfig

    ref_md.Tokenizer.from_pretrained = staticmethod(
        lambda *a, **k: StubTokenizer(cfg.text.vocab_size))
    ref_cfg = RefConfig.from_dict(cfg.to_dict())
    model = ref_md.MoondreamModel(ref_cfg)
    missing, unexpected = model.load_state_dict(state_dict, strict=False)
    persistent_missing = [k for k in missing if "kv_cache" not in k]
    assert not persistent_missing and not unexpected, (persistent_missing, unexpected)
    model.eval()
    return model


def tokens_from_text(text: str) -> List[int]:
    return [int(t) for t in text.split()]


def tensor_sha256(*tensors: torch.Tensor) -> str:
    """sha256 of the raw bytes of the tensors, in order (bit-identity against a stored reference result)"""
    import hashlib

    h = hashlib.sha256()
    for t in tensors:
        h.update(t.detach().contiguous().reshape(-1).view(torch.uint8).numpy().tobytes())
    return h.hexdigest()


def host_arithmetic() -> Dict[str, str]:
    """What decides the bits of the oracle's CPU bf16 results on this host: ATen's vector ISA and the oneDNN kernels
    behind bf16 linear / attention (AMX tiles, AVX-512 bf16, ...), probed on seeded inputs.  The stored reference
    results can only be matched bit for bit on a host where this is the same as on the host that recorded them."""
    import torch.nn.functional as F

    g = torch.Generator().manual_seed(0)
    x, w = (torch.randn(64, 1152, generator=g).to(torch.bfloat16), torch.randn(1152, 1152, generator=g).to(torch.bfloat16))
    q, k, v = (torch.randn(1, 4, 96, 64, generator=g).to(torch.bfloat16) for _ in range(3))
    return {"cpu_capability": torch.backends.cpu.get_cpu_capability(),
            "bf16_probe_sha256": tensor_sha256(F.linear(x, w), F.scaled_dot_product_attention(q, k, v))}
