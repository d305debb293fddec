"""The oracle (CPU restatement of the reference) against the committed golden fixtures produced by the unmodified
reference: replays with the near-tie rule (tests/neartie.py), and bit for bit against reference_bitwise.json."""
import json
import os

import numpy as np
import pytest
import torch

from moondream_b200 import config as C, synth
from oracle import reference_shim as R
from oracle.moondream_oracle import OracleModel

GOLDEN = os.path.join(os.path.dirname(__file__), "golden")


@pytest.fixture(scope="module")
def tiny():
    cfg = C.tiny()
    sd = synth.synthetic_state_dict(cfg, 0)
    return cfg, sd, OracleModel(cfg, sd)


def test_synthetic_weights_are_reproducible(tiny):
    cfg, sd, _ = tiny
    gold = json.load(open(os.path.join(GOLDEN, "synth_hashes.json")))
    assert synth.state_dict_fingerprint(sd, synth.FINGERPRINT_KEYS) == gold["tiny"]
    assert synth.param_count(C.moondream_2b()) == 1_927_237_104      # SURVEY.md appendix A
    assert synth.param_count(C.moondream_0_5b()) == 631_889_382


def test_oracle_reproduces_reference_golden(tiny):
    """replay of the reference-generated fixture on THIS host's CPU: integers exact up to recorded near-ties, floats
    within the host-to-host bf16 accumulation-order spread (tests/neartie.py explains both)"""
    from neartie import MARGIN_ULPS_TOL, check_objects, check_tokens

    cfg, sd, orc = tiny
    gold = json.load(open(os.path.join(GOLDEN, "tiny_reference.json")))
    strict = 0
    for case in gold["cases"]:
        img = synth.synthetic_image(case["image_index"], case["height"], case["width"])
        enc = orc.encode_image(img)
        gen = orc.generate(enc, case["prompt"], len(case["tokens"]))
        n = check_tokens(gen.tokens, case["tokens"], case["margin_ulps"], case["name"])
        strict += n == len(case["tokens"])
        assert np.allclose(gen.margin_ulps[:n], case["margin_ulps"][:n], rtol=0, atol=MARGIN_ULPS_TOL)
        det = orc.generate_points(enc, case["detect_prompt"], True, 3)
        n = check_objects([d["bins"] for d in det], case["detect_bins"], case["detect_ulps"], case["name"] + " detect")
        for d, want in zip(det[:n], case["detect_boxes"]):
            assert all(d[k] == want[k] for k in want)
        pts = orc.generate_points(enc, case["point_prompt"], False, 3)
        n = check_objects([p["bins"] for p in pts], case["point_bins"], case["point_ulps"], case["name"] + " point")
        assert [{"x": p["x"], "y": p["y"]} for p in pts[:n]] == case["points"][:n]
        probe = [float(enc.caches[i][0].float().abs().mean()) for i in (0, cfg.text.n_layers - 1)]
        assert np.allclose(probe, case["kv_abs_mean_first_last"], rtol=1e-3)
    assert strict >= len(gold["cases"]) - 1, "token sequences must reproduce exactly except at most one near-tie flip"


def test_teacher_forcing_is_consistent(tiny):
    cfg, sd, orc = tiny
    img = synth.synthetic_image(5, 378, 378)
    enc = orc.encode_image(img)
    prompt = synth.synthetic_prompt(5, 4, cfg.text.vocab_size)
    free = orc.generate(enc, prompt, 6)
    forced = orc.generate(enc, prompt, 6, forced=free.tokens)
    assert forced.predicted == free.tokens and np.allclose(forced.margins, free.margins)


def test_fp32_truth_is_close_to_bf16_port(tiny):
    cfg, sd, orc = tiny
    truth = OracleModel(cfg, sd, dtype=torch.float32)
    img = synth.synthetic_image(1, 378, 378)
    a = orc.vision_encoder(orc.prepare_crops(img)[0]).float()
    b = truth.vision_encoder(truth.prepare_crops(img)[0])
    assert ((a - b).norm() / b.norm()).item() < 5e-2


def test_oracle_is_bit_identical_to_reference(tiny):
    """encode_image + caption("short") of the unmodified reference (tests/golden/reference_bitwise.json): every layer's
    KV cache bit for bit and the greedy tokens"""
    from neartie import reference_bitwise

    cfg, sd, orc = tiny
    gold = reference_bitwise(exact_bf16=True)["tiny_caption"]
    o_enc = orc.encode_image(synth.synthetic_image(*gold["image"]))
    assert len(o_enc.caches) == cfg.text.n_layers
    assert R.tensor_sha256(*[t for kv in o_enc.caches for t in kv]) == gold["kv_sha256"]
    gen = orc.generate(o_enc, cfg.tokenizer.templates["caption"]["short"], 10)
    assert gen.tokens == gold["tokens"]


def test_oracle_spatial_refs_and_sampling_are_bit_identical_to_reference(tiny):
    """query(spatial_refs=...) (moondream.py:293-301, region.py:96-136): logits and hidden states of the prompt prefill
    with point and box references, then the greedy tokens; and seeded nucleus sampling (moondream.py:270-278)."""
    from neartie import reference_bitwise

    cfg, sd, orc = tiny
    tk = cfg.tokenizer
    gold = reference_bitwise(exact_bf16=True)
    o_enc = orc.encode_image(synth.synthetic_image(*gold["tiny_spatial_refs"]["image"]))
    for c in gold["tiny_spatial_refs"]["cases"]:
        refs = [tuple(r) for r in c["spatial_refs"]]
        prompt = c["prompt"]
        assert prompt.count(tk.coord_id) == 2 * len(refs) and prompt.count(tk.size_id) == sum(len(r) == 4 for r in refs)
        orc.load_encoded(o_enc)
        logits, hidden, _, _ = orc.prefill_prompt(prompt, o_enc.pos, orc.spatial_prompt_embeds(prompt, refs))
        assert R.tensor_sha256(logits) == c["logits_sha256"] and R.tensor_sha256(hidden) == c["hidden_sha256"]
        plain = orc.prefill_prompt(prompt, o_enc.pos)[0]
        assert not torch.equal(plain, logits)                          # the references really enter the prompt
        assert orc.generate(o_enc, prompt, 8, spatial_refs=refs).tokens == c["tokens"]
    sampling = gold["tiny_sampling"]
    assert sampling["image"] == gold["tiny_spatial_refs"]["image"]
    for c in sampling["cases"]:
        torch.manual_seed(c["seed"])
        got = orc.generate(o_enc, sampling["prompt"], 10, temperature=c["temperature"], top_p=c["top_p"]).tokens
        assert got == c["tokens"], c


@pytest.mark.parametrize("preset,head_peak", [("moondream-2b", 3.0), ("moondream-0.5b", 0.0)])
def test_oracle_is_bit_identical_to_reference_on_the_real_architectures(preset, head_peak):
    """The pin on the configurations BASELINE.json quotes, not only on the tiny presets.  Moondream-2B (text 2048 x 24
    layers x 32 heads, ViT 1152 x 27 layers with head_dim 72, vocab 51200) with the bench's synthetic weights (head
    peak 3), its image 0 / prompt 0; and Moondream-0.5B (text 1024 x 16 heads, ViT 720 x 10 heads, MLP width 2690).
    The oracle must reproduce what the UNMODIFIED reference computed (tests/golden/reference_bitwise.json) bit for bit
    on every layer of the 730-token KV prefix, on the greedy tokens and on a 2-object detect."""
    from neartie import reference_bitwise

    gold = reference_bitwise(exact_bf16=True)["real_architectures"][preset]
    assert gold["head_peak"] == head_peak
    cfg = C.preset(preset)
    sd = synth.synthetic_state_dict(cfg, 0, head_peak=head_peak)          # bench.py: HEAD_PEAK = 3 for the 2B
    orc = OracleModel(cfg, sd)
    o_enc = orc.encode_image(synth.synthetic_image(0, 378, 378))
    assert gold["pos"] == o_enc.pos == 730 and len(o_enc.caches) == cfg.text.n_layers
    assert gold["kv_shape"] == [1, cfg.text.n_kv_heads, 730, 64]
    assert all(tuple(t.shape) == tuple(gold["kv_shape"]) for kv in o_enc.caches for t in kv)
    assert R.tensor_sha256(*[t for kv in o_enc.caches for t in kv]) == gold["kv_sha256"]
    prompt = synth.synthetic_prompt(0, 32, cfg.text.vocab_size)     # bench.py: PROMPT_LEN
    gen = orc.generate(o_enc, prompt, 5)
    assert gen.tokens == gold["tokens"]
    # the same five tokens open image 0's caption in every GPU bench run of the round (profiles/r02_bench_final.json:
    # comparators.*.first_tokens, produced by the oracle's arithmetic on the B200)
    if preset == "moondream-2b" and gen.tokens != [1094, 22849, 11037, 121, 36410]:
        assert min(gen.margin_ulps) < 4.5, gen.tokens
    # region head at full width (detect: coordinate + size decode / encode interleaved with decoder steps, moondream.py:653-733)
    tk = cfg.tokenizer
    dprompt = tk.templates["detect"]["prefix"] + [17, 23] + tk.templates["detect"]["suffix"]
    o_det = orc.generate_points(o_enc, dprompt, True, 2)
    det = gold["detect"]
    assert len(o_det) == len(det) and [{k: o[k] for k in d} for o, d in zip(o_det, det)] == det


def test_oracle_reproduces_spatial_ref_golden(tiny):
    """tests/golden/tiny_spatial_refs.json (the reference's query(spatial_refs=...) answers; embedding rows taken after
    bit-equality of the prefill logits with the reference)."""
    from neartie import check_tokens

    cfg, sd, orc = tiny
    gold = json.load(open(os.path.join(GOLDEN, "tiny_spatial_refs.json")))
    idx, h, w = gold["image"]
    o_enc = orc.encode_image(synth.synthetic_image(idx, h, w))
    for c in gold["cases"]:
        refs = [tuple(r) for r in c["spatial_refs"]]
        emb = orc.spatial_prompt_embeds(c["prompt"], refs)
        # one bf16 ulp: the Fourier-feature linear's accumulation order is the host's (tests/neartie.py)
        assert torch.allclose(emb[0, c["rows"]].float(), torch.tensor(c["row_embeds"]), rtol=2 ** -7, atol=1e-6)
        got = orc.generate(o_enc, c["prompt"], len(c["tokens"]), spatial_refs=refs).tokens
        check_tokens(got, c["tokens"], c["margin_ulps"], "spatial refs")
