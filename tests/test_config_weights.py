"""API surface kept from the reference: MoondreamConfig (config.py:5-94) and load_weights_into_model
(weights.py:30-171: safetensors / .pt, canonical keys with optional "model." prefix, legacy HF keys)."""
import json
import os

import pytest
import torch

from moondream_b200 import config as C, synth
from moondream_b200 import weights as W
from moondream_b200.engine import prepare_weights
from oracle.make_golden_bitwise import legacy_dict as _legacy_dict


def test_config_defaults_match_reference_values():
    c = C.MoondreamConfig()
    assert (c.text.dim, c.text.ff_dim, c.text.n_layers, c.text.n_heads, c.text.vocab_size) == (2048, 8192, 24, 32, 51200)
    assert (c.vision.enc_dim, c.vision.enc_ff_dim, c.vision.enc_n_layers, c.vision.enc_n_heads) == (1152, 4304, 27, 16)
    assert (c.vision.crop_size, c.vision.enc_patch_size, c.vision.max_crops, c.vision.overlap_margin) == (378, 14, 12, 4)
    assert c.text.prefix_attn == 730 and c.vision.tokens_per_crop == 729 and c.vision.patch_dim == 588
    assert c.tokenizer.templates["caption"]["normal"] == [1, 32708, 2, 6382, 3]
    assert c.tokenizer.templates["query"] == {"prefix": [1, 15381, 2], "suffix": [3]}
    c.validate()


def test_config_dict_equals_the_reference_config_dict():
    """`MoondreamConfig().to_dict()` (config.py:75-94) key for key against the unmodified reference's
    (tests/golden/reference_bitwise.json), and a dict produced by the reference's config loads into ours (the
    `from_dict` a maintainer would feed with the reference's config JSONs)."""
    from neartie import reference_bitwise

    gold = reference_bitwise()["config"]
    assert C.MoondreamConfig().to_dict() == gold["default"]
    assert C.MoondreamConfig.from_dict(json.loads(json.dumps(gold["default"]))) == C.MoondreamConfig()
    small = json.loads(json.dumps(C.moondream_0_5b().to_dict()))
    assert gold["moondream_0_5b_round_trip"] == small


def test_config_dict_round_trip_and_partial_dict():
    c = C.moondream_0_5b()
    d = json.loads(json.dumps(c.to_dict()))
    assert C.MoondreamConfig.from_dict(d) == c
    part = C.MoondreamConfig.from_dict({"text": {"dim": 1024, "n_heads": 16, "n_kv_heads": 16, "ff_dim": 4096}})
    assert part.text.dim == 1024 and part.vision == C.VisionConfig()


def test_validate_rejects_what_the_kernels_do_not_implement():
    bad = C.MoondreamConfig(text=C.TextConfig(dim=1024, n_heads=16))       # the md05 JSON's missing n_kv_heads
    with pytest.raises(ValueError):
        bad.validate()
    C.MoondreamConfig(text=C.TextConfig(group_size=128)).validate()          # int4 QuantizedLinear blocks (layers.py:54)
    with pytest.raises(ValueError):
        C.MoondreamConfig(text=C.TextConfig(group_size=64)).validate()       # the reference hard-codes 128
    with pytest.raises(ValueError):
        C.preset("no-such-model")


@pytest.mark.parametrize("layout", ["canonical", "model_prefixed", "legacy", "legacy_orig_mod"])
@pytest.mark.parametrize("fmt", ["safetensors", "pt"])
def test_weight_files_load_to_the_canonical_layout(tmp_path, layout, fmt):
    from safetensors.torch import save_file

    cfg = C.tiny()
    sd = synth.synthetic_state_dict(cfg, 1)
    if layout == "canonical":
        tensors = dict(sd)
    elif layout == "model_prefixed":
        tensors = {"model." + k: v for k, v in sd.items()}
    else:
        tensors = _legacy_dict(cfg, sd)
        if layout == "legacy_orig_mod":
            tensors = {k.replace("text_model.", "text_model._orig_mod.", 1): v for k, v in tensors.items()}
    path = str(tmp_path / ("w." + ("safetensors" if fmt == "safetensors" else "pt")))
    if fmt == "safetensors":
        save_file({k: v.contiguous() for k, v in tensors.items()}, path)
    else:
        torch.save(tensors, path)
    loaded = W.load_state_dict_from_file(path, cfg)
    assert set(loaded) == set(sd)
    for k in sd:
        assert loaded[k].dtype == torch.bfloat16 and torch.equal(loaded[k], sd[k]), k


def test_missing_and_misshaped_tensors_are_reported():
    cfg = C.tiny()
    sd = synth.synthetic_state_dict(cfg, 0)
    broken = dict(sd)
    del broken["text.blocks.0.attn.qkv.weight"]
    with pytest.raises(KeyError):
        W.normalize_state_dict(cfg, broken.keys(), broken.__getitem__)
    broken = dict(sd)
    broken["vision.pos_emb"] = torch.zeros(1, 10, 3, dtype=torch.bfloat16)
    with pytest.raises(ValueError):
        W.normalize_state_dict(cfg, broken.keys(), broken.__getitem__)


def test_prepare_weights_pads_for_tma_without_changing_values():
    cfg = C.moondream_0_5b()
    small = C.replace(cfg, vision=C.replace(cfg.vision, enc_n_layers=1), text=C.replace(cfg.text, n_layers=1, vocab_size=64))
    # the geometry checks need prefix_attn etc. unchanged; only depth / vocab shrink so this stays tiny
    sd = synth.synthetic_state_dict(small, 0)
    prepared, patch_k, vis_ff = prepare_weights(small, sd)
    assert patch_k == 592 and vis_ff == 2696 and small.vision.enc_ff_dim == 2690
    keys = [k for k, _, _ in synth.state_dict_spec(small)]
    by = dict(zip(keys, prepared))
    w = by["vision.patch_emb.weight"]
    assert w.shape == (720, 592) and torch.equal(w[:, :588], sd["vision.patch_emb.weight"]) and w[:, 588:].abs().max() == 0
    f1, b1, f2 = by["vision.blocks.0.mlp.fc1.weight"], by["vision.blocks.0.mlp.fc1.bias"], by["vision.blocks.0.mlp.fc2.weight"]
    assert f1.shape == (2696, 720) and b1.shape == (2696,) and f2.shape == (720, 2696)
    assert f1[2690:].abs().max() == 0 and b1[2690:].abs().max() == 0 and f2[:, 2690:].abs().max() == 0
    assert torch.equal(f2[:, :2690], sd["vision.blocks.0.mlp.fc2.weight"])


@pytest.mark.parametrize("layout,fmt", [("legacy", "safetensors"), ("legacy_orig_mod", "pt"), ("model_prefixed", "safetensors"),
                                        ("canonical", "pt")])
def test_loader_agrees_with_the_reference_loader(tmp_path, layout, fmt):
    """The same file went through the unmodified reference's `load_weights_into_model` (weights.py:120-171) into the
    reference model and goes through ours; every parameter must come out identical, which pins the legacy key map (and
    the transposed region feature tensors) to the reference rather than to this repo's reading of it.
    tests/golden/reference_bitwise.json holds what the reference was fed (names, dtypes, shapes and bytes of the file,
    so the file written here must be that file) and the parameters it ended with."""
    from neartie import reference_bitwise

    from oracle.make_golden_bitwise import checkpoint_sha256, weight_file
    from oracle.reference_shim import tensor_sha256

    gold = reference_bitwise()["loader"]
    cfg = C.tiny()
    sd = synth.synthetic_state_dict(cfg, 2)
    path = weight_file(tmp_path, cfg, sd, layout, fmt)
    assert checkpoint_sha256(path) == gold["file_sha256"][f"{layout}-{fmt}"], "not the file the reference loader was fed"
    ours = W.load_state_dict_from_file(path, cfg)
    assert sorted(ours) == sorted(sd) == gold["keys"]
    assert tensor_sha256(*[ours[k] for k in gold["keys"]]) == gold["sha256"][f"{layout}-{fmt}"]
    for k in sd:
        assert torch.equal(ours[k], sd[k]), k


def test_native_safetensors_reader_matches_the_safetensors_package(tmp_path):
    """csrc/loader.cu (mmap + own header parser) against the `safetensors` package the reference loads through
    (weights.py:156-171): names, dtypes, shapes and bytes, with metadata, a scalar, an empty tensor and odd names."""
    import pytest
    from safetensors.torch import save_file

    from moondream_b200 import _native as N
    from moondream_b200.weights import NativeSafetensors

    g = torch.Generator().manual_seed(0)
    tensors = {
        "vision.blocks.0.attn.proj.bias": torch.randn(17, generator=g).to(torch.bfloat16),
        "text.wte": torch.randn(33, 8, generator=g).to(torch.float16),
        'weird "name"/with\\escapes': torch.randn(2, 3, 4, generator=g),
        "ints": torch.arange(10, dtype=torch.int64).view(2, 5),
        "scalar": torch.tensor(3.5),
        "empty": torch.zeros((0, 4), dtype=torch.bfloat16),
        "bytes": torch.arange(7, dtype=torch.uint8),
    }
    path = str(tmp_path / "x.safetensors")
    save_file(tensors, path, metadata={"format": "pt", "note": '{nested: "braces"}'})
    with NativeSafetensors(path) as st:
        assert sorted(st.keys()) == sorted(tensors)
        for k, want in tensors.items():
            got = st.get_tensor(k)
            assert got.dtype == want.dtype and tuple(got.shape) == tuple(want.shape) and torch.equal(got, want), k
    bad = tmp_path / "bad.safetensors"
    bad.write_bytes(b"\xff\xff\xff\xff\x00\x00\x00\x00{}")
    with pytest.raises(N.NativeError):
        NativeSafetensors(str(bad))
    with pytest.raises(N.NativeError):
        NativeSafetensors(str(tmp_path / "missing.safetensors"))


def _st_file(path, header: bytes, payload: bytes = b""):
    import struct

    path.write_bytes(struct.pack("<Q", len(header)) + header + payload)
    return str(path)


def test_native_safetensors_reader_rejects_malformed_and_hostile_headers(tmp_path):
    """A checkpoint is an untrusted file: every malformed header must come back as NativeError — never a crash, a hang,
    or a tensor whose bytes lie outside the mapping."""
    import json

    import pytest

    from moondream_b200 import _native as N
    from moondream_b200.weights import NativeSafetensors

    good = json.dumps({"a": {"dtype": "F32", "shape": [2, 3], "data_offsets": [0, 24]},
                       "__metadata__": {"k": "v", "n": {"deep": [1, 2, {"x": None}]}}}).encode()
    payload = bytes(range(24))
    with NativeSafetensors(_st_file(tmp_path / "good.safetensors", good + b"   ", payload)) as st:     # space padding
        assert st.keys() == ["a"] and st.get_tensor("a").flatten().view(torch.uint8).tolist() == list(payload)
    with NativeSafetensors(_st_file(tmp_path / "nul.safetensors", good + b"\0\0", payload)) as st:
        assert st.keys() == ["a"]

    def entry(**kw):
        e = {"dtype": "F32", "shape": [2, 3], "data_offsets": [0, 24]}
        e.update(kw)
        return {k: v for k, v in e.items() if v is not None}

    hostile = {
        "deep_metadata": b'{"__metadata__": ' + b"[" * 200000 + b"]" * 200000 + b"}",
        "deep_objects": b'{"__metadata__": ' + b'{"a":' * 100000 + b"1" + b"}" * 100000 + b"}",
        "huge_number": b'{"a": {"dtype": "F32", "shape": [' + b"9" * 40 + b'], "data_offsets": [0, 24]}}',
        "huge_offset": b'{"a": {"dtype": "U8", "shape": [1], "data_offsets": [0, 9223372036854775807]}}',
        "negative_dims": json.dumps({"a": entry(shape=[-2, -3])}).encode(),
        "dims_overflow": json.dumps({"a": entry(shape=[2 ** 40, 2 ** 40], dtype="U8", data_offsets=[0, 0])}).encode(),
        "beyond_file": json.dumps({"a": entry(data_offsets=[100, 124])}).encode(),
        "negative_offset": json.dumps({"a": entry(data_offsets=[-8, 16])}).encode(),
        "reversed_offsets": json.dumps({"a": entry(data_offsets=[24, 0])}).encode(),
        "size_mismatch": json.dumps({"a": entry(shape=[2, 2])}).encode(),
        "no_dtype": json.dumps({"a": entry(dtype=None)}).encode(),
        "no_shape": json.dumps({"a": entry(shape=None)}).encode(),
        "no_offsets": json.dumps({"a": entry(data_offsets=None)}).encode(),
        "entry_not_object": b'{"a": [1, 2]}',
        "not_an_object": b'["a"]',
        "trailing_bytes": good + b"}{",
        "unterminated_string": b'{"a',
        "empty": b"",
    }
    for name, header in hostile.items():
        with pytest.raises(N.NativeError):
            NativeSafetensors(_st_file(tmp_path / f"{name}.safetensors", header, payload))
    for cut in range(1, len(good)):                     # every truncation of a valid header
        with pytest.raises(N.NativeError):
            NativeSafetensors(_st_file(tmp_path / "cut.safetensors", good[:cut], payload))
    # a header length that points past the end of the file, and a file shorter than the length field
    (tmp_path / "short.safetensors").write_bytes(b"\x10\x00\x00")
    (tmp_path / "lies.safetensors").write_bytes((1 << 40).to_bytes(8, "little") + good)
    for name in ("short", "lies"):
        with pytest.raises(N.NativeError):
            NativeSafetensors(str(tmp_path / f"{name}.safetensors"))


def test_variant_files_are_found_and_renamed_like_the_reference(tmp_path, monkeypatch):
    """settings["variant"] (row f4): MoondreamModel._lora looks a variant id up in the reference's cache layout
    (lora.py:11-29: $HF_HUB_CACHE/md_variants/<id>/final.pt, else $HF_HOME/hub/...) and applies the reference's key
    renames (lora.py:64-76) to checkpoints saved with the trainer's names.  Compared with what the unmodified
    reference's `variant_state_dict` made of the same file; the expected tree is also spelt out."""
    import pytest

    from moondream_b200 import config as C, synth
    from moondream_b200.moondream import MoondreamModel
    from neartie import reference_bitwise
    from oracle import reference_shim as R
    from oracle.make_golden_bitwise import trainer_named_lora

    cfg = C.tiny()
    flat = synth.synthetic_lora(cfg, 8, 0)                       # canonical names: text.blocks.{i}.{attn.qkv, attn.proj, mlp.fc1, mlp.fc2}.{A, B}
    trainer = trainer_named_lora(flat)                           # the names the trainer saves (what the renames undo)
    assert "text_model.transformer.h.0.mixer.Wqkv.parametrizations.weight.0.A" in trainer
    hub = tmp_path / "hub_cache"
    (hub / "md_variants" / "v1").mkdir(parents=True)
    torch.save(trainer, hub / "md_variants" / "v1" / "final.pt")
    home = tmp_path / "home"
    (home / "hub" / "md_variants" / "v2").mkdir(parents=True)
    torch.save(trainer, home / "hub" / "md_variants" / "v2" / "final.pt")

    seen = []
    model = MoondreamModel(cfg, tokenizer=R.StubTokenizer(cfg.text.vocab_size))
    model._engine = type("E", (), {"load_lora": lambda self, d: seen.append(d) or ("variant", len(seen))})()
    monkeypatch.setenv("HF_HUB_CACHE", str(hub))
    monkeypatch.delenv("HF_HOME", raising=False)
    assert model._lora(None) is None and model._lora({"temperature": 0}) is None
    got = model._lora({"variant": "v1"})
    assert got == ("variant", 1) and model._lora({"variant": "v1"}) is got          # cached per id
    assert sorted(seen[0]) == sorted(flat) and all(torch.equal(seen[0][k], flat[k]) for k in flat)
    with pytest.raises(RuntimeError, match="offline"):
        model._lora({"variant": "v2"})                                              # not in $HF_HUB_CACHE: never downloaded
    monkeypatch.delenv("HF_HUB_CACHE")
    monkeypatch.setenv("HF_HOME", str(home))
    assert model._lora({"variant": "v2"}) == ("variant", 2) and sorted(seen[1]) == sorted(flat)
    assert model._lora({"variant": str(hub / "md_variants" / "v1" / "final.pt")}) == ("variant", 3)   # a path works too
    # the unmodified reference's variant_state_dict("v2") on the same file (tests/golden/reference_bitwise.json)
    def tree_sha256(tree):
        return {k: tree_sha256(v) for k, v in tree.items()} if isinstance(tree, dict) else R.tensor_sha256(tree)

    assert tree_sha256(synth.nest_lora(seen[1])) == reference_bitwise()["variant_tree_sha256"]


def test_lora_variant_table_and_shape_checks():
    """engine.LoraVariant: the per-block (A, B) pointer table the C-ABI takes (md_text_prefill_lora) in the order
    qkv, proj, fc1, fc2, and the errors for adapters that do not fit the model (host logic; tensors on the CPU here)."""
    import pytest

    from moondream_b200 import config as C, synth
    from moondream_b200.engine import LoraVariant

    cfg = C.tiny()
    t = cfg.text
    flat = synth.synthetic_lora(cfg, 8, 0)
    for tree in (synth.nest_lora(flat), synth.nest_lora(flat)["text"]):             # with or without the "text" root
        v = LoraVariant(cfg, tree, "cpu")
        assert v.rank == 8 and len(v.tensors) == t.n_layers * 8 and len(v.table) == t.n_layers * 8
        assert [int(p) for p in v.table] == [x.data_ptr() for x in v.tensors]
        a, b = v.tensors[0], v.tensors[1]                                            # block 0, attn.qkv
        assert tuple(a.shape) == (8, t.dim) and tuple(b.shape) == (3 * t.dim, 8)
        assert torch.equal(a, flat["text.blocks.0.attn.qkv.A"]) and torch.equal(v.tensors[7], flat["text.blocks.0.mlp.fc2.B"])
    bad = dict(flat)
    bad["text.blocks.1.mlp.fc1.B"] = bad["text.blocks.1.mlp.fc1.B"][:-1]            # wrong output width
    with pytest.raises(ValueError, match="block 1 mlp.fc1"):
        LoraVariant(cfg, synth.nest_lora(bad), "cpu")
    with pytest.raises(ValueError, match="multiple of 8"):
        LoraVariant(cfg, synth.nest_lora(synth.synthetic_lora(cfg, 12, 0)), "cpu")
    mixed = dict(flat)
    r16 = synth.synthetic_lora(cfg, 16, 0)
    for k in ("text.blocks.0.attn.proj.A", "text.blocks.0.attn.proj.B"):
        mixed[k] = r16[k]
    with pytest.raises(ValueError, match="share one rank"):
        LoraVariant(cfg, synth.nest_lora(mixed), "cpu")


@pytest.mark.parametrize("preset", ["tiny", "tiny-gqa"])
def test_upload_builds_the_fused_decode_layout_as_views(preset):
    """engine.upload_weights (device = CPU here): per decoder block W1 = [qkv.weight ; fc1.weight], b1 = [qkv.bias ;
    fc1.bias], W2 = [proj.weight | fc2.weight]; the canonical tensors the prefill GEMMs use are VIEWS of those buffers
    (the C runtime checks exactly this adjacency, md_dims.txt_fused), with the checkpoint's values.  With packed
    decoder blocks every block's bf16 pointers alias ONE scratch pair."""
    from moondream_b200 import config as C, synth
    from moondream_b200.engine import upload_weights
    from moondream_b200.synth import state_dict_spec

    cfg = C.preset(preset)
    t = cfg.text
    sd = synth.synthetic_state_dict(cfg, 0)
    keys = [k for k, _, _ in state_dict_spec(cfg)]
    idx = {k: i for i, k in enumerate(keys)}
    prepared, _, _ = prepare_weights(cfg, sd)
    dev, owners = upload_weights(cfg, prepared, "cpu")
    q_rows = t.dim + 2 * t.n_kv_heads * t.head_dim
    for i in range(t.n_layers):
        p = f"text.blocks.{i}."
        qkv, fc1 = dev[idx[p + "attn.qkv.weight"]], dev[idx[p + "mlp.fc1.weight"]]
        proj, fc2 = dev[idx[p + "attn.proj.weight"]], dev[idx[p + "mlp.fc2.weight"]]
        qb, fb = dev[idx[p + "attn.qkv.bias"]], dev[idx[p + "mlp.fc1.bias"]]
        assert tuple(qkv.shape) == (q_rows, t.dim) and qkv.is_contiguous() and fc1.is_contiguous()
        assert fc1.data_ptr() == qkv.data_ptr() + qkv.numel() * 2                   # fc1 rows follow the qkv rows
        assert fb.data_ptr() == qb.data_ptr() + qb.numel() * 2
        assert proj.stride(0) == fc2.stride(0) == t.dim + t.ff_dim                  # column blocks of one matrix
        assert fc2.data_ptr() == proj.data_ptr() + t.dim * 2
        for name, got in (("attn.qkv.weight", qkv), ("mlp.fc1.weight", fc1), ("attn.proj.weight", proj),
                          ("mlp.fc2.weight", fc2), ("attn.qkv.bias", qb), ("mlp.fc1.bias", fb)):
            assert torch.equal(got, sd[p + name]), p + name
    assert all(torch.equal(dev[i], prepared[i]) for i, k in enumerate(keys) if not k.startswith("text.blocks."))
    # packed decoder blocks: bf16 block weights are absent from `prepared` and alias one scratch pair on the device
    prepared_q, _, _ = prepare_weights(cfg, sd, quantized_blocks=True)
    assert all((prepared_q[idx[k]] is None) == k.endswith(("attn.qkv.weight", "attn.proj.weight", "mlp.fc1.weight", "mlp.fc2.weight"))
               for k in keys if k.startswith("text.blocks."))
    dev_q, _ = upload_weights(cfg, prepared_q, "cpu", quantized_blocks=True)
    w1 = {dev_q[idx[f"text.blocks.{i}.attn.qkv.weight"]].data_ptr() for i in range(t.n_layers)}
    w2 = {dev_q[idx[f"text.blocks.{i}.attn.proj.weight"]].data_ptr() for i in range(t.n_layers)}
    assert len(w1) == 1 and len(w2) == 1
    assert torch.equal(dev_q[idx["text.blocks.1.attn.qkv.bias"]], sd["text.blocks.1.attn.qkv.bias"])   # biases stay per block
