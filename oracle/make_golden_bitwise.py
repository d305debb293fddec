"""TEST INFRASTRUCTURE (build container only): what the UNMODIFIED reference computes in the comparisons that pin this
project to it bit for bit, stored so that the tests make them without the reference present.

    python -m oracle.make_golden_bitwise      ->  tests/golden/reference_bitwise.json

Tensors are stored as sha256 of their bytes (oracle.reference_shim.tensor_sha256), token ids, texts and boxes as they
are.  `host` records the CPU arithmetic of the recording host (reference_shim.host_arithmetic): the bf16 results can
only be matched bit for bit where it is the same.  Every input is regenerated from a seed by the tests.
"""
from __future__ import annotations

import json
import os
import sys
import tempfile

import numpy as np
import torch

from moondream_b200 import config as C, synth
from oracle import reference_shim as R

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden", "reference_bitwise.json")
SPATIAL_REFS = ([(0.25, 0.75)], [(0.1, 0.2, 0.5, 0.9)], [(0.25, 0.75), (0.1, 0.2, 0.5, 0.9), (0.6, 0.6)])
SAMPLING = ((5, 0.5, 0.3), (6, 1.5, 0.9))                     # (seed, temperature, top_p)
REAL_ARCHITECTURES = (("moondream-2b", 3.0), ("moondream-0.5b", 0.0))
LOADER_CASES = (("legacy", "safetensors"), ("legacy_orig_mod", "pt"), ("model_prefixed", "safetensors"), ("canonical", "pt"))
INT4_CASES = ((32, 384, True), (128, 128, False), (6, 2048, True))      # (out, in, awkward), seed 100 + index
GQA_CASES = ((0, 378, 378, 5), (1, 500, 700, 9))               # oracle/make_golden_r2.py: (image, h, w, prompt length)
LORA_CASES = ((0, 378, 378, 6), (1, 500, 700, 9))


def kv_sha256(caches) -> str:
    return R.tensor_sha256(*[t for kv in caches for t in kv])


def legacy_dict(cfg, sd):
    """the canonical state dict under the reference's legacy (HF) key names"""
    from moondream_b200 import weights as W

    inv = {v: k for k, v in W.legacy_key_map(cfg).items()}
    out = {inv[k]: v for k, v in sd.items() if k in inv}
    out["region_model.coordinate_features.weight"] = sd["region.coord_features"].T.contiguous()
    out["region_model.size_features.weight"] = sd["region.size_features"].T.contiguous()
    return out


def weight_file(directory, cfg, sd, layout: str, fmt: str) -> str:
    """`sd` written as a checkpoint in one of the layouts the loaders accept"""
    from safetensors.torch import save_file

    if layout == "canonical":
        tensors = dict(sd)
    elif layout == "model_prefixed":
        tensors = {"model." + k: v for k, v in sd.items()}
    else:
        tensors = legacy_dict(cfg, sd)
        if layout == "legacy_orig_mod":
            tensors = {k.replace("text_model.", "text_model._orig_mod.", 1): v for k, v in tensors.items()}
    path = os.path.join(str(directory), "w." + fmt)
    if fmt == "safetensors":
        save_file({k: v.contiguous() for k, v in tensors.items()}, path)
    else:
        torch.save(tensors, path)
    return path


def checkpoint_sha256(path: str) -> str:
    """sha256 over a checkpoint file's (name, dtype, shape, bytes), names sorted, read back with safetensors / torch.load:
    what a loader is fed, independent of the loader"""
    import hashlib

    from safetensors.torch import load_file

    tensors = load_file(path) if path.endswith(".safetensors") else torch.load(path, weights_only=True)
    h = hashlib.sha256()
    for k in sorted(tensors):
        t = tensors[k]
        h.update(f"{k}\0{t.dtype}\0{tuple(t.shape)}\0".encode())
        h.update(t.contiguous().reshape(-1).view(torch.uint8).numpy().tobytes())
    return h.hexdigest()


def trainer_named_lora(flat):
    """a flat canonical LoRA dict under the names the trainer saves (what the reference's renames in lora.py undo)"""
    out = {}
    for k, t in flat.items():
        k2 = (k.replace("text.blocks", "text_model.transformer.h").replace(".attn.qkv", ".mixer.Wqkv")
               .replace(".attn.proj", ".mixer.out_proj"))
        out[k2[:-2] + ".parametrizations.weight.0" + k2[-2:]] = t
    return out


def crop_cases():
    """(image index, h, w, max_crops, margin): ragged sizes, extreme aspect ratios, every max_crops, other margins"""
    rng = np.random.default_rng(123)
    sizes = [(1, 1), (1, 900), (900, 1), (377, 379), (379, 377), (266, 267), (1200, 90)]
    sizes += [(int(rng.integers(2, 1100)), int(rng.integers(2, 1100))) for _ in range(14)]
    cases = []
    for n, (h, w) in enumerate(sizes):
        max_crops = int(rng.integers(1, 13))
        margin = 4 if n % 3 else int(rng.integers(1, 7))
        cases.append((1000 + n, h, w, max_crops, margin))
    return cases


def _tree_sha256(tree):
    return {k: _tree_sha256(v) for k, v in tree.items()} if isinstance(tree, dict) else R.tensor_sha256(tree)


def main():
    assert R.reference_available(), "run where the reference checkout is present"
    from PIL import Image

    if R.REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, R.REFERENCE_ROOT)
    from moondream.torch import lora as ref_lora
    from moondream.torch.config import MoondreamConfig as RefConfig
    from moondream.torch.image_crops import overlap_crop_image as ref_crop
    from moondream.torch.layers import dequantize_tensor as ref_dequantize
    from moondream.torch.rope import precompute_freqs_cis
    from moondream.torch.weights import load_weights_into_model as ref_load

    from moondream_b200 import quant
    from oracle.make_golden_quant import make_case

    torch.manual_seed(0)
    out = {"generator": "oracle/make_golden_bitwise.py (the unmodified reference, CPU, bf16)", "host": R.host_arithmetic()}

    # ---- tiny preset: encode + caption, spatial references, nucleus sampling (moondream.py) ----
    cfg = C.tiny()
    tk = cfg.tokenizer
    sd = synth.synthetic_state_dict(cfg, 0)
    ref = R.load_reference_model(cfg, sd)
    with torch.inference_mode():
        enc = ref.encode_image(Image.fromarray(synth.synthetic_image(11, 600, 450)))
    text = ref.caption(enc, "short", settings={"temperature": 0, "max_tokens": 10})["caption"]
    out["tiny_caption"] = {"image": [11, 600, 450], "kv_sha256": kv_sha256(enc.caches), "tokens": R.tokens_from_text(text)}

    with torch.inference_mode():
        enc = ref.encode_image(Image.fromarray(synth.synthetic_image(2, 500, 700)))
    seen = []
    orig = ref._prefill_prompt

    def recording(prompt_tokens, pos, *a, **k):
        res = orig(prompt_tokens, pos, *a, **k)
        seen.append((prompt_tokens.flatten().tolist(), res[0].clone(), res[1].clone()))
        return res

    ref._prefill_prompt = recording
    spatial = []
    for refs in SPATIAL_REFS:
        seen.clear()
        text = ref.query(enc, "15 16", spatial_refs=refs, settings={"temperature": 0, "max_tokens": 8})["answer"]
        prompt, logits, hidden = seen[0]
        spatial.append({"spatial_refs": [list(r) for r in refs], "prompt": prompt, "logits_sha256": R.tensor_sha256(logits),
                        "hidden_sha256": R.tensor_sha256(hidden), "tokens": R.tokens_from_text(text)})
    ref._prefill_prompt = orig
    prompt = synth.synthetic_prompt(3, 6, cfg.text.vocab_size)
    sampling = []
    for seed, temp, top_p in SAMPLING:
        ref.load_encoded_image(enc)
        torch.manual_seed(seed)
        text = "".join(ref._generate_answer(torch.tensor([prompt]), enc.pos,
                                            {"temperature": temp, "top_p": top_p, "max_tokens": 10}))
        sampling.append({"seed": seed, "temperature": temp, "top_p": top_p, "tokens": R.tokens_from_text(text)})
    out["tiny_spatial_refs"] = {"image": [2, 500, 700], "question": "15 16", "cases": spatial}
    out["tiny_sampling"] = {"image": [2, 500, 700], "prompt": prompt, "cases": sampling}

    # ---- the real architectures, bench weights / inputs ----
    out["real_architectures"] = {}
    for preset, head_peak in REAL_ARCHITECTURES:
        pcfg = C.preset(preset)
        pref = R.load_reference_model(pcfg, synth.synthetic_state_dict(pcfg, 0, head_peak=head_peak))
        with torch.inference_mode():
            penc = pref.encode_image(Image.fromarray(synth.synthetic_image(0, 378, 378)))
        pprompt = synth.synthetic_prompt(0, 32, pcfg.text.vocab_size)
        pref.load_encoded_image(penc)
        text = "".join(pref._generate_answer(torch.tensor([pprompt]), penc.pos, {"temperature": 0, "max_tokens": 5}))
        det = pref.detect(penc, "17 23", settings={"max_objects": 2})["objects"]
        out["real_architectures"][preset] = {
            "head_peak": head_peak, "pos": penc.pos, "kv_shape": list(penc.caches[0][0].shape),
            "kv_sha256": kv_sha256(penc.caches), "tokens": R.tokens_from_text(text), "detect": det}
        del pref, penc

    # ---- grouped-query decoder and LoRA variant (the cases of oracle/make_golden_r2.py) ----
    gcfg = C.tiny_gqa()
    gref = R.load_reference_model(gcfg, synth.synthetic_state_dict(gcfg, 0))
    gqa = []
    for idx, h, w, _ in GQA_CASES:
        with torch.inference_mode():
            gqa.append(kv_sha256(gref.encode_image(Image.fromarray(synth.synthetic_image(idx, h, w))).caches))
    hub = tempfile.mkdtemp()
    os.environ["HF_HUB_CACHE"] = hub
    os.makedirs(os.path.join(hub, "md_variants", "synthetic-r8"))
    torch.save(synth.synthetic_lora(cfg, rank=8, seed=0), os.path.join(hub, "md_variants", "synthetic-r8", "final.pt"))
    lora = []
    for idx, h, w, _ in LORA_CASES:
        with torch.inference_mode():
            lenc = ref.encode_image(Image.fromarray(synth.synthetic_image(idx, h, w)),
                                    {"temperature": 0, "variant": "synthetic-r8"})
        lora.append(kv_sha256(lenc.caches))
    out["round2_kv_sha256"] = {"tiny_gqa": gqa, "tiny_lora": lora}

    # ---- host tables, config, loaders, int4, crops ----
    out["rope_sha256"] = {}
    for preset in ("tiny", "moondream-2b"):
        t = C.preset(preset).text
        out["rope_sha256"][preset] = R.tensor_sha256(precompute_freqs_cis(t.dim // (2 * t.n_heads), t.max_context))
    out["config"] = {"default": RefConfig().to_dict(),
                     "moondream_0_5b_round_trip": RefConfig.from_dict(C.moondream_0_5b().to_dict()).to_dict()}

    # per layout: the file the reference's loader was fed (checkpoint_sha256) and the parameters it left in its model
    # (names, and one sha256 over them in name order)
    out["loader"] = {"file_sha256": {}, "sha256": {}}
    lsd = synth.synthetic_state_dict(cfg, 2)
    for layout, fmt in LOADER_CASES:
        model = R.load_reference_model(cfg, synth.synthetic_state_dict(cfg, 5))      # different weights: overwritten
        path = weight_file(tempfile.mkdtemp(), cfg, lsd, layout, fmt)
        ref_load(path, model)
        theirs = {k: v for k, v in model.state_dict().items() if "kv_cache" not in k}
        assert out["loader"].setdefault("keys", sorted(theirs)) == sorted(theirs)
        out["loader"]["file_sha256"][f"{layout}-{fmt}"] = checkpoint_sha256(path)
        out["loader"]["sha256"][f"{layout}-{fmt}"] = R.tensor_sha256(*[theirs[k] for k in sorted(theirs)])

    home = tempfile.mkdtemp()
    os.makedirs(os.path.join(home, "hub", "md_variants", "v2"))
    torch.save(trainer_named_lora(synth.synthetic_lora(cfg, 8, 0)), os.path.join(home, "hub", "md_variants", "v2", "final.pt"))
    os.environ.pop("HF_HUB_CACHE")
    os.environ["HF_HOME"] = home
    ref_lora.variant_state_dict.cache_clear()
    out["variant_tree_sha256"] = _tree_sha256(ref_lora.variant_state_dict("v2"))

    out["int4_dequant"] = []
    for seed, (o, i, awk) in enumerate(INT4_CASES):
        nib, scale, zero = make_case(100 + seed, o, i, awk)
        want = ref_dequantize(quant.pack_reference_int4(nib), scale.reshape(-1, 1), zero.reshape(-1, 1), (o, i), torch.bfloat16)
        out["int4_dequant"].append(R.tensor_sha256(want))

    out["crops"] = []
    for idx, h, w, max_crops, margin in crop_cases():
        theirs = ref_crop(synth.synthetic_image(idx, h, w), overlap_margin=margin, max_crops=max_crops)
        out["crops"].append({"tiling": list(theirs["tiling"]), "sha256": R.tensor_sha256(torch.from_numpy(theirs["crops"]))})

    json.dump(out, open(OUT, "w"), indent=1)
    print("wrote", OUT)


if __name__ == "__main__":
    main()
