"""Host-built tables the kernels consume: the 256-entry pixel LUT (reference vision.py:33-40) and the RoPE table
(rope.py:6-17 as text.py:215-219 calls it).  Both must be bit-identical to what the reference computes."""
import numpy as np
import torch

from moondream_b200 import config as C
from moondream_b200.engine import pixel_lut, rope_table
from oracle import reference_shim as R


def test_pixel_lut_is_the_reference_normalisation():
    from oracle.moondream_oracle import OracleModel
    from moondream_b200 import synth

    lut = pixel_lut()
    assert lut.dtype == torch.bfloat16 and lut.shape == (256,)
    assert float(lut[0]) == -1.0 and float(lut[255]) == 1.0 and bool((lut[1:] >= lut[:-1]).all())
    # through the oracle's prepare_crops (bit-identical to the reference's, tests/test_oracle.py): an image holding
    # every byte value, no resize (378 x 378)
    cfg = C.tiny()
    orc = OracleModel(cfg, synth.synthetic_state_dict(cfg, 0))
    img = (np.arange(378 * 378 * 3, dtype=np.int64) % 256).astype(np.uint8).reshape(378, 378, 3)
    crops = orc.prepare_crops(img)[0]                       # bf16 [n, 3, 378, 378]
    want = lut[torch.from_numpy(img).long()].permute(2, 0, 1)
    assert torch.equal(crops[0], want)


def test_rope_table_is_the_reference_table():
    """against precompute_freqs_cis of the unmodified reference (tests/golden/reference_bitwise.json)"""
    from neartie import reference_bitwise

    gold = reference_bitwise()["rope_sha256"]
    for preset in ("tiny", "moondream-2b"):
        t = C.preset(preset).text
        mine = rope_table(t.head_dim, t.max_context)
        assert mine.dtype == torch.float32 and tuple(mine.shape) == (t.max_context, t.head_dim // 4, 2)
        assert R.tensor_sha256(mine) == gold[preset], preset
