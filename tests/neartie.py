"""Comparison helpers for the CPU tests that replay committed fixtures (tests/golden/*.json) through the oracle.

The fixtures were produced by the unmodified reference on ONE host.  torch's CPU bf16 matmuls go through oneDNN, whose
accumulation order depends on the ISA it dispatches (AMX tiles on the fixture host and on the GPU boxes, AVX-512 bf16
emulation on hosts without AMX), so a second host reproduces the reference's logits only to a couple of bf16 ulps: the
fixtures' margins move by <= 2 ulps and an argmax whose recorded margin is 0-1 ulp may flip.  Bit-identity with the
reference is therefore asserted LIVE (oracle and reference in one process: test_oracle.py::*bit_identical*,
test_oracle_r2.py::test_round2_restatements_*), and fixture replays use the same near-tie rule as the GPU parity tests
(tests/test_model_parity_gpu.py): integers exact, except that a decision may differ where the fixture's own recorded
top-1/top-2 margin is below NEAR_TIE_ULPS bf16 ulps, after which that sequence legitimately diverges and its comparison stops.
"""
from __future__ import annotations

import math

NEAR_TIE_ULPS = 4.5          # same threshold and derivation as tests/test_model_parity_gpu.py
MARGIN_ULPS_TOL = 4.0        # two bf16 evaluations of one margin: observed <= 2 ulps between AMX and AVX-512 hosts


def check_tokens(got, want, want_ulps, what=""):
    """exact match, or first divergence at a recorded near-tie; returns the number of leading tokens that agree"""
    assert len(got) == len(want) or any(u < NEAR_TIE_ULPS for u in want_ulps), (what, len(got), len(want))
    for i, (g, w) in enumerate(zip(got, want)):
        if g != w:
            assert want_ulps[i] < NEAR_TIE_ULPS, f"{what}: token {i}: {g} vs {w} at a recorded margin of {want_ulps[i]} ulps"
            return i
    return min(len(got), len(want))


def check_objects(got_bins, want_bins, want_ulps, what=""):
    """region-head bins per object (x, y[, w, h]) plus the continue/stop decision (last entry of each ulps row);
    returns the number of leading objects that agree in every bin"""
    for n, (wb, wu) in enumerate(zip(want_bins, want_ulps)):
        assert n < len(got_bins), f"{what}: object {n} missing"
        for j, (g, w) in enumerate(zip(got_bins[n], wb)):
            if g != w:
                assert wu[j] < NEAR_TIE_ULPS, f"{what}: object {n} bin {j}: {g} vs {w} at {wu[j]} ulps"
                return n
        if wu[-1] < NEAR_TIE_ULPS:
            return n + 1
    assert len(got_bins) == len(want_bins), f"{what}: {len(got_bins)} objects vs {len(want_bins)}"
    return len(want_bins)


def reference_bitwise(exact_bf16: bool = False) -> dict:
    """tests/golden/reference_bitwise.json (oracle/make_golden_bitwise.py): what the unmodified reference computed.
    `exact_bf16`: the caller compares CPU bf16 results bit for bit, which only a host with the recording host's CPU
    arithmetic can reproduce (see above); elsewhere the test is skipped and the fixture replays stand in for it."""
    import json
    import os

    import pytest

    from oracle import reference_shim as R

    gold = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_bitwise.json")))
    if exact_bf16 and R.host_arithmetic() != gold["host"]:
        pytest.skip(f"this host's CPU bf16 arithmetic {R.host_arithmetic()} is not the recording host's {gold['host']}")
    return gold


def json_close(got, want, float_tol, path=""):
    """structural equality of two JSON values: ints / strings / bools / shapes exact, floats within
    float_tol(path) where path is the key path with list indices dropped.  Returns a list of mismatches."""
    bad = []
    if isinstance(want, dict):
        if not isinstance(got, dict) or got.keys() != want.keys():
            return [f"{path}: keys differ"]
        for k in want:
            bad += json_close(got[k], want[k], float_tol, f"{path}/{k}")
    elif isinstance(want, list):
        if not isinstance(got, list) or len(got) != len(want):
            return [f"{path}: length {len(got) if isinstance(got, list) else got!r} vs {len(want)}"]
        for g, w in zip(got, want):
            bad += json_close(g, w, float_tol, path)
    elif isinstance(want, float) or isinstance(got, float):
        if got is None or want is None or isinstance(got, (str, bool)) or isinstance(want, (str, bool)):
            bad.append(f"{path}: {got!r} vs {want!r}")
        elif not (math.isclose(got, want, rel_tol=0.0, abs_tol=float_tol(path)) or got == want):
            bad.append(f"{path}: {got} vs {want} (tol {float_tol(path)})")
    elif got != want:
        bad.append(f"{path}: {got!r} vs {want!r}")
    return bad
