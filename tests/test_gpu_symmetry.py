"""-m gpu: USE_SYMMETRY engine mode (SURVEY 8f/f4).

The reference has two symmetric jump rules behind its compile-time switch; the engine implements both (include/kgx.h):
  "lastjump": the device rule (GPUCompute.h:53-58), which Kangaroo::Check replays on the CPU (Check.cpp:534-556): jump = x mod 32
              bumped when it repeats the kangaroo's previous jump;
  "symclass": the rule of the working symmetric path, SolveKeyCPU (Kangaroo.cpp:381-384, 422-428): x mod 16 + 16 * symClass.
Both: P += J, d += jD mod n, class switch (y > (p-1)/2 -> y = p - y, d = n - d).  Restated in oracle/kgx_oracle.c
(kgo_jump_sym), pinned to the reference's Int / IntGroup code by tests/test_oracle_vs_ref.py.  Checked here
  * through the C ABI on every jump kernel (state + DP multiset, several launches so lastJump persists across launches),
  * through the reference's UNMODIFIED host compiled with -DUSE_SYMMETRY and linked to the engine (oracle/_ref/kangaroo_b200_sym):
    its own `-check` prints CPU/GPU ok (KGX_SYM_RULE=lastjump) -- which the reference's own symmetric GPU kernel cannot
    (DESIGN.md, symmetry) -- and in64 is solved with the default symclass rule,
  * statistically: operations per solved key with and without symmetry (the reference's -DSTATS counters), ~1/sqrt(2)."""
import os
import re
import subprocess

import numpy as np
import pytest

from kangaroo_b200 import GPUEngine, NB_RUN
from oracle import kgo

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")


@pytest.fixture(autouse=True)
def _no_symmetric_tmem_kernel(request):
    if "kernel" in request.fixturenames and request.getfixturevalue("kernel").get("kernel") == "tmem":
        pytest.skip("the TMEM tile kernel has no symmetric instantiation")


def sym_case(oracle, n, rp=64, seed=1, first_type=0):
    table = oracle.create_jump_table_sym(rp)
    key = oracle.ec_mul_g(0x5B3F38AF935A3640D158E871CE6E9666DB862636383386EE0000000000123000)
    wdiv4 = ((1 << rp) - 1) >> 2
    oracle.rseed(seed)
    px, py, d = oracle.create_herd_sym(n, rp, wdiv4, key, first_type)
    return dict(table=table, key=key, px=px, py=py, d=d, n=n, rp=rp)


RULES = [("lastjump", 32), ("symclass", 0)]


@pytest.mark.parametrize("rule,init", RULES, ids=[r for r, _ in RULES])
@pytest.mark.parametrize("grid", [(2, 4), (3, 5), (16, 8)])
def test_symmetric_walk_matches_oracle(oracle, kernel, grid, rule, init):
    n = grid[0] * grid[1] * 128
    case = sym_case(oracle, n, seed=grid[0] * 10 + grid[1])
    eng = GPUEngine(grid[0], grid[1], 0, 1 << 17, **kernel)
    eng.SetSymmetry(rule)
    mask = oracle.dp_mask(7)
    eng.SetParams(mask, *case["table"])
    eng.SetWildOffset(((1 << 64) - 1) >> 2)            # what the host passes (Kangaroo.cpp:548-550); not applied in this mode
    eng.SetKangaroos(case["px"], case["py"], kgo.array_to_ints(case["d"]))
    px, py, d = case["px"].copy(), case["py"].copy(), case["d"].copy()
    lj = np.full(n, init, dtype=np.uint8)
    eng.callKernel()
    for launch in range(3):                            # lastJump / symClass must survive between launches
        found = eng.Launch()
        want = oracle.jump_sym(px, py, d, lj, case["table"], NB_RUN, mask, grp=256, max_dp=1 << 20, rule=rule)
        assert sorted((it.x, it.d, it.kIdx) for it in found) == sorted((x, dd, k) for x, dd, k, j in want), launch
        assert len(found) > 0
    want = oracle.jump_sym(px, py, d, lj, case["table"], NB_RUN, mask, grp=256, max_dp=1 << 20, rule=rule)     # launch 4 is in flight
    gx, gy, gd = eng.GetKangaroos()
    assert gx == kgo.array_to_ints(px) and gy == kgo.array_to_ints(py) and gd == kgo.array_to_ints(d)
    half = (kgo.P - 1) // 2
    assert max(gy) <= half                             # every point is its class representative
    assert any(v > kgo.N // 2 for v in gd)             # negative distances were exercised
    eng.sync(); eng.close()


@pytest.mark.parametrize("rule,init", RULES, ids=[r for r, _ in RULES])
def test_symmetric_set_kangaroo_resets_rule_state(oracle, kernel, rule, init):
    """SetKangaroo stores lastJump = NB_JUMP (GPUEngine.cu:532-536) / symClass = 0 for the patched kangaroo."""
    n = 2 * 2 * 128
    case = sym_case(oracle, n, seed=5)
    eng = GPUEngine(2, 2, 0, 1 << 16, **kernel)
    eng.SetSymmetry(rule)
    mask = oracle.dp_mask(16)
    eng.SetParams(mask, *case["table"])
    eng.SetKangaroos(case["px"], case["py"], kgo.array_to_ints(case["d"]))
    px, py, d = case["px"].copy(), case["py"].copy(), case["d"].copy()
    lj = np.full(n, init, dtype=np.uint8)
    eng.callKernel(); eng.Launch(relaunch=False)
    oracle.jump_sym(px, py, d, lj, case["table"], NB_RUN, mask, rule=rule)
    r = 77
    oracle.rseed(31337)
    nx, ny, nd = oracle.create_herd_sym(1, 64, ((1 << 64) - 1) >> 2, case["key"], r % 2)
    px[r], py[r], d[r], lj[r] = nx[0], ny[0], nd[0], init
    eng.SetKangaroo(r, kgo.from_limbs(nx[0]), kgo.from_limbs(ny[0]), kgo.from_limbs(nd[0]))
    eng.callKernel(); eng.Launch(relaunch=False)
    oracle.jump_sym(px, py, d, lj, case["table"], NB_RUN, mask, rule=rule)
    gx, gy, gd = eng.GetKangaroos()
    assert gx == kgo.array_to_ints(px) and gy == kgo.array_to_ints(py) and gd == kgo.array_to_ints(d)
    eng.close()


def test_symmetric_device_herd_matches_reference_formula(oracle, kernel):
    """kgx_create_herd in symmetric mode == Kangaroo::CreateHerd's USE_SYMMETRY branch (Kangaroo.cpp:686-734)."""
    n = 2 * 128
    case = sym_case(oracle, n, seed=9)
    # the oracle's d already carries the class switch; recover the drawn distances by undoing it where y was flipped
    key = case["key"]
    raw = []
    for i in range(n):
        dv = kgo.from_limbs(case["d"][i])
        pt = oracle.ec_mul_g(dv) if i % 2 == 0 else oracle.ec_add(key, oracle.ec_mul_g(dv))
        raw.append(dv if pt[1] == kgo.from_limbs(case["py"][i]) else (kgo.N - dv) % kgo.N)
    eng = GPUEngine(2, 1, 0, 65536, **kernel)
    eng.SetSymmetry("symclass")
    eng.CreateHerd(raw, key)
    gx, gy, gd = eng.GetKangaroos()
    assert gx == kgo.array_to_ints(case["px"]) and gy == kgo.array_to_ints(case["py"]) and gd == kgo.array_to_ints(case["d"])
    eng.close()


def test_symmetric_device_hash_convert(oracle, kernel):
    """kgx_convert_dps in symmetric mode: the record's distance is a signed 128-bit value (no wild offset); the 40-byte DP
    must equal HashTable::Convert(x, d mod n, type) (HashTable.cpp:75-100)."""
    import torch
    from kangaroo_b200.dist import SlabView, decode_dp40
    n = 2 * 4 * 128
    case = sym_case(oracle, n, seed=21)
    eng = GPUEngine(2, 4, 0, 65536, **kernel)
    eng.SetSymmetry("symclass")
    eng.SetParams(oracle.dp_mask(5), *case["table"])
    eng.SetKangaroos(case["px"], case["py"], kgo.array_to_ints(case["d"]))
    eng.callKernel()
    found = eng.Launch(relaunch=False)
    ptr = eng.convert_dps_device_ptr()
    raw = torch.as_tensor(SlabView(ptr, 4 + 65536 * 40), device="cuda").cpu()
    cnt = int.from_bytes(bytes(raw[:4].numpy().tobytes()), "little")
    assert cnt == len(found) > 100
    want = {}
    for it in found:
        h, X, D = oracle.hash_convert(it.x, it.d, it.kIdx % 2)
        want[(it.kIdx & 0xFFFFFFFF, X)] = (h, D)
    n_neg = 0
    for kidx, h, x, dist, ktype in decode_dp40(raw[4:4 + cnt * 40]):
        D = (abs(dist) & ((1 << 126) - 1)) | ((1 << 127) if dist < 0 else 0) | (ktype << 126)
        assert (h, D) == want[(kidx, x)]
        n_neg += dist < 0
    assert n_neg > 0
    eng.close()


def run(binary, args, timeout=900, env=None, cwd=None):
    exe = os.path.join(ROOT, "oracle", "_ref", binary)
    if not os.path.exists(exe):
        pytest.skip("oracle/_ref/%s not built (needs the reference sources at build time)" % binary)
    e = dict(os.environ); e.update(env or {})
    p = subprocess.run([exe] + args, capture_output=True, text=True, timeout=timeout, cwd=cwd or ROOT, env=e)
    return (p.stdout + p.stderr).replace("\r", "\n")


@pytest.mark.parametrize("env", [{"KGX_MODE": "stream", "KGX_STREAM_G": "128"}, {"KGX_MODE": "resident"}], ids=["stream128", "resident"])
def test_reference_check_with_use_symmetry(env):
    """The reference host compiled with its own USE_SYMMETRY switch, its own Check.cpp:467-621 replay (which follows the DEVICE
    rule: lastJump), our engine switched to that rule."""
    env = dict(env, KGX_SYM_RULE="lastjump")
    out = run("kangaroo_b200_sym", ["-gpu", "-check", "-g", "8,128"], env=env)
    assert "CPU/GPU ok" in out, out[-3000:]
    assert "DP Mismatch" not in out and "not ok" not in out


def test_symmetric_build_solves_in64():
    """Default rule of the symmetric drop-in = symclass (the rule SolveKeyCPU runs).  With the lastjump rule the same program
    does not terminate on this input: kangaroos fall into fruitless cycles longer than two (measured, DESIGN.md)."""
    out = run("kangaroo_b200_sym", ["-t", "0", "-gpu", "-g", "64,128", os.path.join(GOLD, "in64.txt")], timeout=300)
    assert "5B3F38AF935A3640D158E871CE6E9666DB862636383386EE510F18CCC3BD72EB" in out.upper(), out[-2000:]


def test_symmetry_gain_in_operations_per_key(tmp_path):
    """64 keys in a 2^56 range, the reference's -DSTATS counters: average group operations per solved key in units of sqrt(N),
    without and with symmetry (theory 2.08 vs 1.47, ComputeExpected, Kangaroo.cpp:836-873).  Every key must be solved by both
    builds; the averages are recorded."""
    cfg = os.path.join(GOLD, "in56_64keys.txt")
    avgs = {}
    for binary in ("kangaroo_b200_stats", "kangaroo_b200_sym_stats"):
        # 65,536 kangaroos, dp 9: DP overhead nK * 2^dp = 3.4e7 << sqrt(N) = 2.7e8, ~8 k DPs per launch (dp 4 floods the 131072-record
        # buffer and the host table: the first attempt ran at 240 MK/s, host-bound)
        out = run(binary, ["-t", "0", "-gpu", "-g", "4,128", "-d", "9", cfg], timeout=600, cwd=str(tmp_path))
        rows = re.findall(r"^\[\s*(\d+)\] 2\^([0-9.]+) Dead:(\d+) Avg:2\^([0-9.]+) DeadAvg:[0-9.]+ \(([0-9.]+) ([0-9.]+) sqrt\(N\)\)", out, re.M)
        assert len(rows) == 64, out[-2000:]
        assert out.count("Priv: 0x") == 64
        avgs[binary] = (float(rows[-1][4]), float(rows[-1][5]))
        print("%s: avg %.3f sqrt(N) per key (expected %.3f)" % (binary, *avgs[binary]))
    plain, sym = avgs["kangaroo_b200_stats"][0], avgs["kangaroo_b200_sym_stats"][0]
    # Measured on a B200: 2.23 vs 1.90 sqrt(N) (ratio 0.85) and 2.00 vs 1.98 (0.99) in two runs (profiles/r2_symmetry_gain.txt).
    # The ideal 1/sqrt(2) does not materialise in the reference's symmetric walk at all: its own CPU-only build (no engine
    # involved) gives 2.30 vs 2.17 sqrt(N) over 96 keys of a 2^44 range (ratio 0.95, 25 dead kangaroos per key instead of 1.6).
    # So this is a record + sanity bound (64-key averages scatter by ~9 %), not a claim of the theoretical gain.
    assert sym < 1.25 * plain, avgs
    with open(str(tmp_path / "symmetry_gain.txt"), "w") as f:
        f.write("64 keys, 2^56 range, grid 4x128 (65,536 kangaroos), dp 9, reference host (-DSTATS) + B200 engine\n")
        f.write("plain    : %.3f sqrt(N) operations per key (reference's estimate %.3f)\n" % avgs["kangaroo_b200_stats"])
        f.write("symmetry : %.3f sqrt(N) operations per key (reference's estimate %.3f)\n" % avgs["kangaroo_b200_sym_stats"])
        f.write("ratio    : %.3f (theory 0.707)\n" % (sym / plain))
