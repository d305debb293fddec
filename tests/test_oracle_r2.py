"""CPU: the oracle's round-2 restatements against the fixtures the UNMODIFIED reference produced
(oracle/make_golden_r2.py): grounded reasoning (moondream.py:323-432), text-only query (:565-574), a grouped-query
decoder (text.py:36-38,49) and `_apply_top_p` (:270-278)."""
import json
import os

import pytest
import torch

from neartie import check_objects, check_tokens

HERE = os.path.dirname(os.path.abspath(__file__))


def _gold(name):
    return json.load(open(os.path.join(HERE, "golden", name)))


@pytest.fixture(scope="module")
def tiny():
    from moondream_b200 import config as C, synth

    cfg = C.tiny()
    return cfg, synth.synthetic_state_dict(cfg, 0)


def test_reasoning_matches_the_reference(tiny):
    from moondream_b200 import synth
    from oracle.moondream_oracle import OracleModel

    cfg, sd = tiny
    from neartie import NEAR_TIE_ULPS, check_tokens

    gold = _gold("tiny_reasoning.json")
    sd = dict(sd)
    sd["text.lm_head.bias"] = synth.special_token_bias(sd, cfg, *gold["bias"])
    orc = OracleModel(cfg, sd)
    saw_coord = saw_answer = False
    for c in gold["cases"]:
        enc = orc.encode_image(synth.synthetic_image(c["image_index"], c["height"], c["width"]))
        r = orc.generate_reasoning(enc, c["prompt"], c["max_tokens"])
        n = check_tokens(r["tokens"], c["reasoning_tokens"], c["margin_ulps"] + [c["end_margin_ulps"]], "reasoning")
        if n < len(c["reasoning_tokens"]) or r["coords"] != c["coords"]:
            # a flip at a recorded near-tie (token or coordinate bin): the chain legitimately diverges from there
            flips = [u for u in c["margin_ulps"] + [x for x in c["coord_ulps"] if x is not None] if u < NEAR_TIE_ULPS]
            assert flips, ("reasoning", r["tokens"], c["reasoning_tokens"], r["coords"], c["coords"])
            continue
        ans = orc.generate(None, cfg.tokenizer.templates["query"]["suffix"], c["max_tokens"], pos=r["pos"])
        check_tokens(ans.tokens, c["answer_tokens"], c["answer_margin_ulps"], "answer")
        saw_coord |= sum(t == cfg.tokenizer.coord_id for t in r["tokens"]) >= 2
        saw_answer |= len(r["tokens"]) < c["max_tokens"]
    assert saw_coord and saw_answer, "the fixture must exercise the coordinate interleave and the answer_id stop"


def test_text_only_query_matches_the_reference(tiny):
    from oracle.moondream_oracle import OracleModel

    cfg, sd = tiny
    gold = _gold("tiny_text_only.json")
    orc = OracleModel(cfg, sd)
    for c in gold["cases"]:
        check_tokens(orc.generate(None, c["prompt"], c["max_tokens"]).tokens, c["tokens"], c["margin_ulps"], "text-only")
    # the causal mask matters: the same prompt under the prefix-LM mask gives other hidden states
    c = gold["cases"][2]
    orc.reset_cache()
    a = orc.prefill_prompt(c["prompt"], 0, causal=True)[1]
    orc.reset_cache()
    b = orc.prefill_prompt(c["prompt"], 0, causal=False)[1]
    assert not torch.equal(a, b)


def test_gqa_decoder_matches_the_reference():
    from moondream_b200 import config as C, synth
    from oracle.moondream_oracle import OracleModel

    cfg = C.tiny_gqa()
    cfg.validate()
    sd = synth.synthetic_state_dict(cfg, 0)
    assert sd["text.blocks.0.attn.qkv.weight"].shape == (256 + 2 * 2 * 64, 256)
    orc = OracleModel(cfg, sd)
    for c in _gold("tiny_gqa.json")["cases"]:
        enc = orc.encode_image(synth.synthetic_image(c["image_index"], c["height"], c["width"]))
        assert tuple(enc.caches[0][0].shape) == (1, 2, 730, 64)
        check_tokens(orc.generate(enc, c["prompt"], len(c["tokens"])).tokens, c["tokens"], c["margin_ulps"], "gqa/lora")


def test_lora_variant_matches_the_reference(tiny):
    from moondream_b200 import synth
    from oracle.moondream_oracle import OracleModel

    cfg, sd = tiny
    gold = _gold("tiny_lora.json")
    orc = OracleModel(cfg, sd)
    orc.lora = synth.nest_lora(synth.synthetic_lora(cfg, gold["rank"], gold["seed"]))
    for c in gold["cases"]:
        enc = orc.encode_image(synth.synthetic_image(c["image_index"], c["height"], c["width"]))
        check_tokens(orc.generate(enc, c["prompt"], len(c["tokens"])).tokens, c["tokens"], c["margin_ulps"], "gqa/lora")
        det = orc.generate_points(enc, c["detect_prompt"], True, 2)
        check_objects([o["bins"] for o in det], c["detect_bins"], c["detect_ulps"], "lora detect")
    orc.lora = None
    enc = orc.encode_image(synth.synthetic_image(0, 378, 378))
    assert orc.generate(enc, gold["cases"][0]["prompt"], 12).tokens != gold["cases"][0]["tokens"]   # the adapters matter


def test_apply_top_p_matches_the_reference():
    from moondream_b200.sampling import apply_top_p

    for c in _gold("top_p.json")["cases"]:
        logits = torch.tensor(c["logits"]).to(torch.bfloat16).unsqueeze(0)
        probs = torch.softmax(logits / c["temperature"], dim=-1)
        kept = apply_top_p(probs, c["top_p"])
        nz = kept[0].nonzero().flatten().tolist()
        assert nz == c["kept_ids"]
        assert kept[0, nz].float().tolist() == c["kept_probs"]


def test_round2_restatements_are_bit_identical_to_the_reference_here(tiny):
    """Every case of oracle/make_golden_r2.py through the oracle, on a host with the recording host's CPU arithmetic:
    what the unmodified reference returned must come out exactly (reasoning texts and grounding, answers, tokens,
    detected boxes; every layer's KV cache bit for bit, tests/golden/reference_bitwise.json), and the oracle's own
    recorded margins, logits and probes within the host-to-host accumulation-order spread (tests/neartie.py)."""
    from moondream_b200 import config as C, synth
    from neartie import MARGIN_ULPS_TOL, json_close, reference_bitwise
    from oracle import reference_shim as R
    from oracle.make_golden_r2 import _grounding_from
    from oracle.moondream_oracle import OracleModel

    kv_sha = reference_bitwise(exact_bf16=True)["round2_kv_sha256"]
    cfg, sd = tiny
    tk = cfg.tokenizer
    stub = R.StubTokenizer(cfg.text.vocab_size)

    def tol(path):
        if path.endswith("ulps"):
            return MARGIN_ULPS_TOL
        if path.endswith("/logits"):
            return 0.25                       # 2 bf16 ulps at |logit| <= 16
        return 2e-3                           # KV probes (means of |k|)

    def close(got, case, what):
        bad = json_close(got, {k: case[k] for k in got}, tol)
        assert not bad, (what, bad[:5])

    def kv(enc):
        return R.tensor_sha256(*[t for pair in enc.caches for t in pair])

    def probe(enc, last):
        return [float(enc.caches[i][0].float().abs().mean()) for i in (0, last)]

    def reasoning(orc, enc, prompt, max_tokens):
        r = orc.generate_reasoning(enc, prompt, max_tokens)
        ans = orc.generate(None, tk.templates["query"]["suffix"], max_tokens, pos=r["pos"])
        return r, ans, {"reasoning_tokens": r["tokens"], "coords": r["coords"], "margin_ulps": r["margin_ulps"],
                        "coord_ulps": r["coord_ulps"], "end_margin_ulps": r["end_margin_ulps"],
                        "answer_tokens": ans.tokens, "answer_margin_ulps": ans.margin_ulps}

    gold = _gold("tiny_reasoning.json")
    sd_r = dict(sd)
    sd_r["text.lm_head.bias"] = synth.special_token_bias(sd, cfg, *gold["bias"])
    orc_r = OracleModel(cfg, sd_r)
    for c in gold["cases"]:
        enc = orc_r.encode_image(synth.synthetic_image(c["image_index"], c["height"], c["width"]))
        r, ans, got = reasoning(orc_r, enc, c["prompt"], c["max_tokens"])
        assert _grounding_from(r["tokens"], r["coords"], tk, stub.decode) == (c["reasoning_text"], c["grounding"])
        assert ans.tokens == R.tokens_from_text(c["answer"])
        close(got, c, "reasoning")

    gold = _gold("tiny_text_only.json")
    orc = OracleModel(cfg, sd)
    for c in gold["cases"]:
        gen = orc.generate(None, c["prompt"], c["max_tokens"])
        close({"tokens": gen.tokens, "margin_ulps": gen.margin_ulps}, c, "text-only")
    c = gold["reasoning"]
    close(reasoning(orc_r, None, c["prompt"], c["max_tokens"])[2], c, "text-only reasoning")

    gcfg = C.tiny_gqa()
    gorc = OracleModel(gcfg, synth.synthetic_state_dict(gcfg, 0))
    for c, want in zip(_gold("tiny_gqa.json")["cases"], kv_sha["tiny_gqa"]):
        enc = gorc.encode_image(synth.synthetic_image(c["image_index"], c["height"], c["width"]))
        assert kv(enc) == want
        gen = gorc.generate(enc, c["prompt"], len(c["tokens"]))
        close({"tokens": gen.tokens, "margin_ulps": gen.margin_ulps,
               "kv_abs_mean_first_last": probe(enc, gcfg.text.n_layers - 1)}, c, "gqa")

    gold = _gold("tiny_lora.json")
    orc.lora = synth.nest_lora(synth.synthetic_lora(cfg, gold["rank"], gold["seed"]))
    for c, want in zip(gold["cases"], kv_sha["tiny_lora"]):
        enc = orc.encode_image(synth.synthetic_image(c["image_index"], c["height"], c["width"]))
        assert kv(enc) == want
        gen = orc.generate(enc, c["prompt"], len(c["tokens"]))
        det = orc.generate_points(enc, c["detect_prompt"], True, 2)
        assert len(det) == len(c["detect_boxes"]) and [{k: o[k] for k in d} for o, d in zip(det, c["detect_boxes"])] == c["detect_boxes"]
        close({"tokens": gen.tokens, "margin_ulps": gen.margin_ulps, "detect_bins": [o["bins"] for o in det],
               "detect_ulps": [o["ulps"] for o in det], "kv_abs_mean_first_last": probe(enc, cfg.text.n_layers - 1)},
              c, "lora")
    orc.lora = None

    # _apply_top_p's inputs: the oracle's prefill logits on image 0 (its kept sets are test_apply_top_p_matches_the_reference)
    enc = orc.encode_image(synth.synthetic_image(0, 378, 378))
    for c in _gold("top_p.json")["cases"]:
        orc.load_encoded(enc)
        close({"logits": orc.prefill_prompt(c["prompt"], enc.pos)[0][0].float().tolist()}, c, "top_p")
