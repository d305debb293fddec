"""Host-side pieces of bench.py that need no GPU: the FLOP model behind `roofline` / `step_model_tflops` against the
survey's figures (SURVEY.md §8d), the nvidia-smi clock parser, and the one-JSON-line stdout guard."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def test_flop_model_matches_the_survey():
    import bench
    from moondream_b200 import config as C

    cfg2b = C.preset("moondream-2b")
    # SURVEY.md §8d: per image 3.514 TF with 2 crops, 8.845 TF with 10, 10.84 TF with 13 (2B, 32-token prompt, 64 new)
    for crops, tf in ((2, 3.514), (10, 8.845), (13, 10.84)):
        got = bench.flops_per_image(cfg2b, crops) / 1e12
        assert abs(got - tf) / tf < 0.01, (crops, got, tf)
    got = bench.flops_per_image(C.preset("moondream-0.5b"), 2) / 1e12
    assert abs(got - 1.147) / 1.147 < 0.02, got


def test_clock_sampler_parses_nvidia_smi_lines():
    import bench

    s = bench.ClockSampler(0)
    s.proc = type("P", (), {"terminate": lambda self: None, "wait": lambda self, timeout=None: 0, "kill": lambda self: None})()
    s.lines = ["1965, 1965, 400.1, Not Active, Not Active, Not Active, Not Active",
               "1575, 1965, 990.0, Not Active, Not Active, Not Active, Active",
               "1590, 1965, 985.2, Not Active, Not Active, Not Active, Active",
               "210, 1965, 150.0, Not Active, Not Active, Not Active, Not Active",     # idle sample: ignored by the median
               "garbage"]
    out = s.stop()
    assert out["sm_max_mhz"] == 1965.0 and out["reasons"] == ["sw_power_cap"] and out["samples"] == 4
    assert out["sm_mhz"] == 1590.0


def test_stdout_carries_exactly_one_json_line():
    code = ("import bench, os; bench.protect_stdout(); os.write(1, b'NCCL version banner\\n'); print('library chatter'); "
            "bench.emit_line({'metric': 'x', 'value': 1.0})")
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, cwd=ROOT, timeout=300)
    assert r.returncode == 0, r.stderr[-500:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1 and json.loads(lines[0]) == {"metric": "x", "value": 1.0}
    assert "NCCL version banner" in r.stderr and "library chatter" in r.stderr


def test_reference_arm_exits_quietly_on_other_ranks():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    r = subprocess.run([sys.executable, "bench.py", "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, cwd=ROOT, env=env, timeout=300)
    assert r.returncode == 0 and r.stdout.strip() == "", (r.returncode, r.stdout[-300:], r.stderr[-300:])


def _gate(monkeypatch, free_rows, forced_rows, oracle_tokens, oracle_ulps):
    """bench.parity_gate with the CPU oracle and the engine replaced by stand-ins that return the given tokens."""
    import torch

    import bench

    gens = {}
    for g, (toks, ulps) in enumerate(zip(oracle_tokens, oracle_ulps)):
        gens[g] = type("Gen", (), {"tokens": list(toks), "predicted": list(toks), "margin_ulps": list(ulps)})()
    monkeypatch.setattr(bench, "cpu_sample", lambda cfg, sd, index, n: (1.0, {"image": index}, gens[index]))
    monkeypatch.setattr(bench, "cpu_threads", lambda: 1)

    class Eng:
        def encode_crops_with_prompt(self, crops, offsets, tilings, prompts):
            return ["prefix"] * len(prompts), "hidden"

        def generate(self, prefixes, prompts, max_tokens, forced=None, **kw):
            assert forced is not None and all(forced[i][:-1] == list(oracle_tokens[i]) for i in range(len(oracle_tokens)))
            return type("R", (), {"tokens": torch.tensor(forced_rows, dtype=torch.int32)})()

    prompts = [[1, 2, 3]] * len(free_rows)
    check = [(i, i) for i in range(len(oracle_tokens))]
    return bench.parity_gate(None, None, Eng(), None, None, None, prompts, torch.tensor(free_rows, dtype=torch.int32), check)


def test_parity_gate_accepts_near_tie_flips_and_rejects_clear_mismatches(monkeypatch):
    """The gate that decides whether bench.py may print a value: a divergence is tolerated only where the ORACLE's own
    top-1 / top-2 margin is below 4.5 bf16 ulps; a disagreement at a clear margin — free-running or teacher-forced —
    fails it."""
    import bench

    n = bench.NEW_TOKENS
    base = [[100 + s for s in range(n)], [200 + s for s in range(n)]]
    wide = [[30.0] * n, [30.0] * n]
    pad = lambda rows: [r + [0] for r in rows]                       # the engine returns max_tokens + 1 slots
    # 1. identical outputs
    rep, cpu = _gate(monkeypatch, pad(base), pad(base), base, wide)
    assert rep["ok"] and rep["free_running_first_divergence"] == [None, None] and rep["free_running_strict_sequences"] == "2/2"
    assert rep["teacher_forced"] == {"steps": 2 * n, "strict_agree": 2 * n, "steps_with_margin_ge_near_tie": 2 * n, "agree_on_those": 2 * n}
    assert cpu["kind"] == "port" and cpu["cores"] == 1
    # 2. a flip where the oracle itself is at a 1-ulp margin: tolerated, reported
    ulps = [list(wide[0]), list(wide[1])]
    ulps[1][7] = 1.0
    free = [list(base[0]), list(base[1])]
    free[1][7:] = [999] * (n - 7)                                    # legitimately diverged from step 7 on
    forced = [list(base[0]), list(base[1])]
    forced[1][7] = 999
    rep, _ = _gate(monkeypatch, pad(free), pad(forced), base, ulps)
    assert rep["ok"] and rep["free_running_first_divergence"] == [None, 7] and rep["free_running_strict_sequences"] == "1/2"
    assert rep["teacher_forced"]["strict_agree"] == 2 * n - 1 and rep["teacher_forced"]["agree_on_those"] == 2 * n - 1
    # 3. the same flip at a clear margin: the gate fails (free-running)
    rep, _ = _gate(monkeypatch, pad(free), pad(base), base, wide)
    assert not rep["ok"] and "image 1 diverges at step 7" in rep["error"]
    # 4. free-running happens to agree but a teacher-forced step disagrees at a clear margin: fails too
    rep, _ = _gate(monkeypatch, pad(base), pad(forced), base, wide)
    assert not rep["ok"] and "teacher-forced" in rep["error"]


def test_dump_outputs_writes_the_token_ids_as_float32(tmp_path):
    import numpy as np
    import torch

    import bench

    tokens = torch.tensor([[1, 51199, 0], [7, 8, 9]], dtype=torch.int32)
    bench.dump_outputs(str(tmp_path / "out"), tokens)
    got = np.load(tmp_path / "out" / "tokens.npy")
    assert got.dtype == np.float32 and np.array_equal(got, tokens.numpy())


@pytest.mark.parametrize("argv,flag", [(["--steps", "0"], "--steps"),
                                       (["--impl", "reference", "--dump-outputs", "out"], "--dump-outputs")])
def test_arguments_bench_cannot_honour_are_rejected(tmp_path, argv, flag):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + argv, capture_output=True, text=True,
                       cwd=tmp_path, timeout=300)
    assert r.returncode == 2 and flag in r.stderr and r.stdout.strip() == ""
    assert not (tmp_path / "out").exists()
