"""CPU (no GPU needed): BASELINE config 1 -- the reference's unmodified host program linked against the engine's GPUEngine
shim still runs its CPU-only mode (SolveKeyCPU plumbing, `-t N`, no device touched).  First five keys of
VC_CUDA8/in40_1000.txt; expected private keys from SURVEY.md section 4 (reference CPU run)."""
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "oracle", "_ref", "kangaroo_b200")
EXPECTED = ["57004A31CED094F0", "57004A31D2F397AF", "57004A00A71C8425", "57004A73420E46DF", "57004ACEF20EBCFD"]


def test_in40_cpu_only_through_dropin_binary():
    if not os.path.exists(BIN):
        pytest.skip("oracle/_ref/kangaroo_b200 not built (needs the reference sources at build time)")
    p = subprocess.run([BIN, "-t", "2", os.path.join(ROOT, "tests", "golden", "in40_5.txt")], capture_output=True, text=True,
                       timeout=600, cwd=ROOT)
    out = (p.stdout + p.stderr).upper()
    for k in EXPECTED:
        assert "62CE27C8FED90758A834C2CB6E3F19BC8A0B5E7D92C0FC0F" + k in out, out[-1500:]
    assert "FAILED" not in out
