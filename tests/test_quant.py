"""Weight-only int8 groundwork (BASELINE.json config 5; SURVEY.md §8c: int8 parity = the bf16 path on the dequantised
weights).  CPU only: format invariants, error bound, and the drift the oracle sees on dequantised weights."""
import pytest
import torch

from moondream_b200 import config as C, quant, synth


def test_round_trip_bounds_and_edge_rows():
    g = torch.Generator().manual_seed(0)
    w = (torch.randn(96, 320, generator=g) * 0.05).to(torch.bfloat16)
    w[3] = 0                                          # an all-zero output feature
    w[5, 7] = 2.0                                     # an outlier sets that row's scale
    q, s = quant.quantize_weight_int8(w)
    assert q.dtype == torch.int8 and s.dtype == torch.bfloat16 and q.shape == w.shape and s.shape == (96,)
    assert int(q.abs().max()) <= 127 and bool((s.float() > 0).all())
    d = quant.dequantize_weight_int8(q, s)
    assert d.dtype == torch.bfloat16 and bool((d[3] == 0).all())
    # |w - w'| <= half a quantisation step + one bf16 rounding of the product (2^-9 relative)
    err = (w.float() - d.float()).abs()
    bound = 0.5 * s.float().unsqueeze(1) * (1 + 2 ** -7) + d.float().abs() * 2 ** -8
    assert bool((err <= bound).all()), float((err - bound).max())
    # every row uses (almost) its whole range: the row maximum quantises to +-127 or +-126 (bf16 scale rounding)
    rowmax = q.abs().amax(dim=1)
    assert bool((rowmax[torch.arange(96) != 3] >= 126).all())
    # idempotent: re-quantising the dequantised weights reproduces q and scale
    q2, s2 = quant.quantize_weight_int8(d)
    assert torch.equal(s2, s) and torch.equal(q2, q)
    with pytest.raises(ValueError):
        quant.quantize_weight_int8(torch.zeros(4))


def test_decoder_packing_and_stream_bytes():
    cfg = C.tiny()
    sd = synth.synthetic_state_dict(cfg, 0)
    packed, deq = quant.quantize_decoder_int8(cfg, sd)
    keys = list(quant.decode_stream_keys(cfg))
    assert set(packed) == set(keys) and len(keys) == 4 * cfg.text.n_layers + 1
    for k in sd:
        if k in packed:
            assert deq[k].shape == sd[k].shape and deq[k].dtype == torch.bfloat16 and not torch.equal(deq[k], sd[k])
        else:
            assert deq[k] is sd[k]                     # vision, embeddings, norms, biases, region head untouched
    big = C.preset("moondream-2b")
    bf16, i8 = quant.stream_bytes(big, False), quant.stream_bytes(big, True)
    assert abs(bf16 / 1e9 - 2.63) < 0.02               # SURVEY.md §8d: 2.63 GB per decode step
    assert 0.50 < i8 / bf16 < 0.51


def test_oracle_drift_on_dequantised_weights():
    """The int8 oracle is the bf16 oracle on w'; report how far it moves from the unquantised model."""
    from oracle.moondream_oracle import OracleModel

    cfg = C.tiny()
    sd = synth.synthetic_state_dict(cfg, 0)
    _, deq = quant.quantize_decoder_int8(cfg, sd)
    a, b = OracleModel(cfg, sd), OracleModel(cfg, deq)
    img = synth.synthetic_image(3, 378, 378)
    prompt = synth.synthetic_prompt(3, 6, cfg.text.vocab_size)
    ea, eb = a.encode_image(img), b.encode_image(img)
    # the image prefix runs through the (quantised) decoder blocks: KV drifts, the vision tower does not
    k0a, k0b = ea.caches[0][0].float(), eb.caches[0][0].float()
    rel = float((k0a - k0b).norm() / k0a.norm())
    assert 0 < rel < 5e-2, rel
    la = a.prefill_prompt(prompt, ea.pos)[0].float()
    b.load_encoded(eb)
    lb = b.prefill_prompt(prompt, eb.pos)[0].float()
    assert float((la - lb).norm() / la.norm()) < 0.1


# ---------------------------------------------------------------------------------------------------------------
# int4 group-128: the reference's QuantizedLinear checkpoint format (layers.py:38-110)
# ---------------------------------------------------------------------------------------------------------------
import hashlib
import json
import os

HERE = os.path.dirname(os.path.abspath(__file__))


def _sha(t):
    return hashlib.sha256(t.contiguous().view(torch.int16).numpy().tobytes()).hexdigest()


def test_int4_dequantisation_matches_the_reference_vectors():
    """tests/golden/int4_dequant.json holds hashes of what the UNMODIFIED `dequantize_tensor` (layers.py:38-44) returned
    (oracle/make_golden_quant.py); the oracle restatement and the product-side formula must reproduce them."""
    from oracle.make_golden_quant import make_case
    from oracle.moondream_oracle import dequantize_tensor

    gold = json.load(open(os.path.join(HERE, "golden", "int4_dequant.json")))
    assert len(gold["cases"]) >= 5
    for c in gold["cases"]:
        nib, scale, zero = make_case(c["seed"], c["out"], c["in"], c["awkward"])
        packed = quant.pack_reference_int4(nib)
        assert packed.shape == (c["out"] * c["in"] // 256, 128) and packed.dtype == torch.uint8
        orc = dequantize_tensor(packed, scale.reshape(-1, 1), zero.reshape(-1, 1), (c["out"], c["in"]))
        assert _sha(orc) == c["sha256"] and orc.flatten()[:16].view(torch.int16).tolist() == c["first16"]
        mine = quant.dequantize(quant.unpack_reference_int4(packed, c["out"], c["in"]), scale, zero)
        assert _sha(mine) == c["sha256"]


def test_int4_against_the_reference_function_when_present():
    """against dequantize_tensor of the unmodified reference (layers.py:38-44, tests/golden/reference_bitwise.json)"""
    from neartie import reference_bitwise

    from oracle.make_golden_bitwise import INT4_CASES
    from oracle.make_golden_quant import make_case
    from oracle.reference_shim import tensor_sha256

    gold = reference_bitwise()["int4_dequant"]
    assert len(gold) == len(INT4_CASES) == 3
    for seed, ((o, i, awk), want) in enumerate(zip(INT4_CASES, gold)):
        nib, scale, zero = make_case(100 + seed, o, i, awk)
        assert tensor_sha256(quant.dequantize(nib, scale, zero)) == want


def test_int4_layout_round_trips_and_error_bound():
    g = torch.Generator().manual_seed(5)
    w = (torch.randn(48, 384, generator=g) * 0.03).to(torch.bfloat16)
    nib, scale, zero = quant.quantize_weight_int4(w)
    assert nib.dtype == torch.uint8 and int(nib.max()) <= 15 and scale.shape == zero.shape == (48, 3)
    assert torch.equal(quant.unpack_reference_int4(quant.pack_reference_int4(nib), 48, 384), nib)
    st = quant.to_stream_int4(nib)
    assert st.shape == (48, 192)
    assert torch.equal(st & 15, nib[:, 0::2]) and torch.equal(st >> 4, nib[:, 1::2])
    d = quant.dequantize(nib, scale, zero)
    err = (w.float() - d.float()).abs().view(48, 3, 128)
    # half a step (+ the bf16 rounding of scale and of the product) inside the group's range
    assert bool((err <= 0.52 * scale.unsqueeze(-1) + d.float().abs().view(48, 3, 128) * 2 ** -8 + 1e-6).all())
    with pytest.raises(ValueError):
        quant.quantize_weight_int4(torch.zeros(4, 100))
    with pytest.raises(ValueError):
        quant.unpack_reference_int4(torch.zeros(3, 128, dtype=torch.uint8), 48, 384)


@pytest.mark.parametrize("bits", [4, 8])
def test_quantize_decoder_and_reference_checkpoint_round_trip(bits):
    cfg = C.tiny()
    sd = synth.synthetic_state_dict(cfg, 0)
    qt, deq = quant.quantize_decoder(cfg, sd, bits)
    assert qt.bits == bits and len(qt.blocks) == cfg.text.n_layers
    t = cfg.text
    w1q, w1s, w1z, w2q, w2s, w2z = qt.fused(1)
    rows1 = t.dim + 2 * t.n_kv_heads * t.head_dim + t.ff_dim
    assert w1q.shape == (rows1, t.dim * bits // 8) and w1s.shape == w1z.shape == (rows1, t.dim // 128)
    assert w2q.shape == (t.dim, (t.dim + t.ff_dim) * bits // 8) and w2s.shape == (t.dim, (t.dim + t.ff_dim) // 128)
    for k in sd:
        if k.startswith("text.blocks.") and k.endswith(("qkv.weight", "proj.weight", "fc1.weight", "fc2.weight")):
            assert deq[k].dtype == torch.bfloat16 and deq[k].shape == sd[k].shape
            assert 0 < float((deq[k].float() - sd[k].float()).norm() / sd[k].float().norm()) < (0.2 if bits == 4 else 0.02)
        else:
            assert deq[k] is sd[k]
    if bits == 8:
        # the int8 scheme of round 1 (one bf16 scale per row) is the zero = 0, repeated-scale case of the shared formula
        q8, s8 = quant.quantize_weight_int8(sd["text.blocks.0.mlp.fc1.weight"])
        assert torch.equal(quant.dequantize_weight_int8(q8, s8), deq["text.blocks.0.mlp.fc1.weight"])
        return
    # a checkpoint in the reference's format loads back to the same quantised state and the same dequantised weights
    ck = {k: v for k, v in sd.items() if k not in deq or deq[k] is sd[k]}
    ck.update(quant.reference_checkpoint_entries(cfg, qt))
    assert quant.is_quantized_checkpoint(ck) and not quant.is_quantized_checkpoint(sd)
    qt2, rest = quant.from_reference_checkpoint(cfg, ck)
    for a, b in zip(qt.blocks, qt2.blocks):
        for name in a:
            assert torch.equal(a[name].values, b[name].values) and torch.equal(a[name].scale, b[name].scale)
    from oracle.moondream_oracle import dequantized_state_dict

    orc_sd = dequantized_state_dict(ck)
    for k in deq:
        assert torch.equal(orc_sd[k], deq[k]), k
    assert set(rest) == {k for k in sd if k not in deq or deq[k] is sd[k]}


def test_stream_bytes_accounting():
    big = C.preset("moondream-2b")
    bf16 = quant.stream_bytes(big)
    assert 0.30 < quant.stream_bytes(big, bits=4) / bf16 < 0.34        # blocks / 4 + scales, LM head bf16
    assert 0.54 < quant.stream_bytes(big, bits=8) / bf16 < 0.58


def test_loader_passes_reference_int4_entries_through(tmp_path):
    """weights.load_state_dict_from_file keeps `…weight.packed / .scale / .zero_point` (layers.py:58-76) as they are —
    uint8 / fp32, no bf16 cast, no shape check against the dense layout — and still normalises everything else."""
    from moondream_b200 import weights

    cfg = C.tiny()
    sd = synth.synthetic_state_dict(cfg, 0)
    qt, deq = quant.quantize_decoder(cfg, sd, 4)
    ck = {k: v for k, v in sd.items() if deq[k] is sd[k]}
    ck.update(quant.reference_checkpoint_entries(cfg, qt))
    ck = {"model." + k: v for k, v in ck.items()}                 # the reference's optional prefix (weights.py:123-131)
    path = str(tmp_path / "int4.pt")
    torch.save(ck, path)
    loaded = weights.load_state_dict_from_file(path, cfg)
    assert quant.is_quantized_checkpoint(loaded)
    k = "text.blocks.2.mlp.fc1.weight"
    assert k not in loaded and loaded[k + ".packed"].dtype == torch.uint8 and loaded[k + ".scale"].dtype == torch.float32
    assert loaded["text.blocks.2.mlp.fc1.bias"].dtype == torch.bfloat16 and loaded["vision.pos_emb"].dtype == torch.bfloat16
    qt2, rest = quant.from_reference_checkpoint(cfg, loaded)
    assert torch.equal(qt2.blocks[2]["mlp.fc1"].dequantized(), deq[k])
    with pytest.raises(KeyError):                                  # a dense matrix that is neither present nor packed
        bad = dict(ck)
        bad.pop("model.text.blocks.1.attn.proj.weight.packed")
        torch.save(bad, path)
        weights.load_state_dict_from_file(path, cfg)
