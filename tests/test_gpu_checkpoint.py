"""-m gpu: work-file walks on the device (kgx_walks_*: export, import, verification) and the solver's checkpoint / resume
(kangaroo_b200/solver.py --work-file / --work-interval / --save-kangaroos / --resume)."""
import os
import re
import signal
import subprocess
import sys
import time

import numpy as np
import pytest

from kangaroo_b200 import GPUEngine, NB_RUN
from kangaroo_b200 import ecmath as ec
from kangaroo_b200.ingest import read_work_info
from oracle import kgo
from tests.gpu_util import make_case, expected_after

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")
REFBIN = os.path.join(ROOT, "oracle", "_ref", "kangaroo_ref_cpu")
DROPIN = os.path.join(ROOT, "oracle", "_ref", "kangaroo_b200")
PRIV110 = "35C0D7234DF7DEB0F20CF7062444"


def _records(px, py, d):
    """(n, 12) work-file records from int lists (d unbiased mod n)"""
    return np.concatenate([kgo.ints_to_array(px), kgo.ints_to_array(py), kgo.ints_to_array(d)], axis=1).astype(np.uint64)


def _engine(case, kernel, groups=2, tpg=2, sym=None):
    eng = GPUEngine(groups, tpg, 0, 1 << 16, **kernel)
    if sym:
        eng.SetSymmetry(sym)
    eng.SetParams(case["mask"], *case["table"])
    eng.SetWildOffset(case["wdiv2"])
    return eng


def _case(oracle, n, seed=21):
    c = make_case(oracle, n, range_power=64, seed=seed)
    c["mask"] = oracle.dp_mask(6)
    return c


def _launches(eng, k):
    dps = []
    for _ in range(k):
        eng.callKernel()
        dps += [(it.x, it.d, it.kIdx) for it in eng.Launch(relaunch=False)]
    return dps


@pytest.mark.parametrize("sym", [None, "lastjump", "symclass"])
def test_export_equals_get_kangaroos(oracle, kernel, sym):
    if sym and kernel.get("kernel") == "tmem":
        pytest.skip("the TMEM tile kernel has no symmetric instantiation")
    n = 512
    case = _case(oracle, n)
    eng = _engine(case, kernel, sym=sym)
    eng.SetKangaroos(case["px"], case["py"], kgo.array_to_ints(case["d"]))
    _launches(eng, 2)
    recs = eng.GetWalks()
    px, py, d = eng.GetKangaroos()
    assert np.array_equal(recs, _records(px, py, d))
    wild_neg = sum(1 for i in range(1, n, 2) if d[i] > kgo.N // 2)
    assert wild_neg > 0 or sym                                       # the n - |d| form is exercised
    eng.close()


def test_continuation_is_bit_exact(oracle, kernel):
    n, k, m = 512, 2, 3
    case = _case(oracle, n)
    a = _engine(case, kernel)
    a.SetKangaroos(case["px"], case["py"], kgo.array_to_ints(case["d"]))
    _launches(a, k)
    recs = a.GetWalks()
    b = _engine(case, kernel)
    assert b.LoadWalks(recs, key=case["key"])[0] == 0
    assert np.array_equal(b.GetWalks(), recs)
    da, db = _launches(a, m), _launches(b, m)
    assert np.array_equal(a.GetWalks(), b.GetWalks()) and sorted(da) == sorted(db)
    ex, ey, ed, edps = expected_after(oracle, case, m * NB_RUN, case["mask"], px=np.ascontiguousarray(recs[:, 0:4]),
                                      py=np.ascontiguousarray(recs[:, 4:8]), d=np.ascontiguousarray(recs[:, 8:12]))
    assert np.array_equal(b.GetWalks(), np.concatenate([ex, ey, ed], axis=1).astype(np.uint64))
    assert sorted(db) == edps
    a.close(); b.close()


def test_continuation_across_geometries(oracle, kernel):
    """two engines of n walks -> one engine of 2n on another kernel: the same walks continue identically"""
    n, m = 512, 2
    case = _case(oracle, 2 * n, seed=33)
    halves = []
    for h in range(2):
        e = _engine(case, kernel)
        e.SetKangaroos(case["px"][h * n:(h + 1) * n], case["py"][h * n:(h + 1) * n], kgo.array_to_ints(case["d"][h * n:(h + 1) * n]))
        _launches(e, 1)
        halves.append(e)
    recs = np.concatenate([e.GetWalks() for e in halves])
    other = dict(kernel="resident") if kernel.get("kernel") != "resident" else dict(kernel="stream", stream_g=8)
    big = _engine(case, other, groups=2, tpg=4)
    assert big.nbKangaroo == 2 * n
    assert big.LoadWalks(recs, key=case["key"])[0] == 0
    d_small = [_launches(e, m) for e in halves]
    d_big = _launches(big, m)
    assert np.array_equal(big.GetWalks(), np.concatenate([e.GetWalks() for e in halves]))
    assert sorted(d_big) == sorted(d_small[0] + [(x, d, k + n) for x, d, k in d_small[1]])
    for e in halves + [big]:
        e.close()


def test_verify_flags_exactly_the_corrupted_records(oracle):
    n = 512
    case = _case(oracle, n, seed=44)
    eng = _engine(case, dict(kernel="stream"))
    eng.CreateHerd(kgo.array_to_ints(case["d"]), case["key"])
    _launches(eng, 1)
    recs = eng.GetWalks()
    bad = recs.copy()
    bad[6, 4] ^= np.uint64(1 << 17)                                  # one bit of y, tame
    bad[9, 8] += np.uint64(1)                                        # wild distance off by one
    nb, idx = eng.LoadWalks(bad, key=case["key"])
    assert nb == 2 and list(idx) == [6, 9]
    other = ec.mul(0x1234567890ABCDEF)
    nb, idx = eng.LoadWalks(recs, key=other)                         # the whole herd against another key: every wild walk
    assert nb == n // 2 and list(idx) == list(range(1, n, 2))
    assert eng.LoadWalks(recs, key=case["key"])[0] == 0
    eng.close()


def test_verify_full_size_herd(capsys):
    from kangaroo_b200 import random_herd_arrays
    eng = GPUEngine(296, 128, 0, 1 << 16)
    n = eng.nbKangaroo
    assert n == 4849664
    key = ec.mul(0x1234567)
    eng.SetWildOffset(1 << 79)
    sc, d128 = random_herd_arrays(n, 80, 1 << 79, np.random.Generator(np.random.PCG64(5)))
    eng.CreateHerdRaw(sc, d128, key)
    t0 = time.perf_counter()
    recs = eng.GetWalks()
    t1 = time.perf_counter()
    nb, _ = eng.LoadWalks(recs, key=key)
    t2 = time.perf_counter()
    assert nb == 0
    with capsys.disabled():
        print("\n[walks] %d walks: export + copy %.3f s, import + verify %.3f s" % (n, t1 - t0, t2 - t1))
    eng.close()


def test_partial_import_leaves_the_rest(oracle, kernel):
    n = 512
    case = _case(oracle, n, seed=55)
    eng = _engine(case, kernel)
    eng.SetKangaroos(case["px"], case["py"], kgo.array_to_ints(case["d"]))
    before = eng.GetWalks()
    other = _case(oracle, n, seed=56)
    new = _records(kgo.array_to_ints(other["px"]), kgo.array_to_ints(other["py"]), kgo.array_to_ints(other["d"]))
    c = 200
    assert eng.LoadWalks(new[:c], key=other["key"])[0] == 0
    after = eng.GetWalks()
    assert np.array_equal(after[:c], new[:c]) and np.array_equal(after[c:], before[c:])
    with pytest.raises(RuntimeError, match="herd"):
        eng.LoadWalks(np.concatenate([new, new[:2]]), key=other["key"])
    eng.close()


# ---- the solver --------------------------------------------------------------------------------------------------------
def solver(args, timeout=900):
    p = subprocess.run([sys.executable, "-m", "kangaroo_b200.solver"] + args, capture_output=True, text=True, timeout=timeout, cwd=ROOT)
    return p.stdout + p.stderr


GRID, NK = "32,128", 32 * 128 * 128


@pytest.fixture(scope="module")
def saved(tmp_path_factory):
    """puzzle110_window64 stopped after K steps with a checkpoint of table and kangaroos"""
    work = str(tmp_path_factory.mktemp("ck") / "p110.work")
    k = 12
    out = solver([os.path.join(GOLD, "puzzle110_window64.txt"), "--dp", "10", "--grid", GRID, "--seed", "5", "--max-steps", str(k),
                  "--work-file", work, "--save-kangaroos"])
    assert PRIV110 not in out, "the key was found before the checkpoint: pick a smaller --max-steps\n" + out[-2000:]
    assert "Key# 0 not found" in out and "checkpoint: " + work in out, out[-2000:]
    return work, k, out


def test_solver_checkpoint_file(saved):
    work, k, _ = saved
    info = read_work_info(work)
    assert info.n_walks == NK and os.path.getsize(work) == info.walk_offset + 96 * NK
    assert info.total_count == (k + 1) * NK * NB_RUN                  # K steps + the launch in flight at the stop
    assert not os.path.exists(work + ".tmp")
    if os.path.exists(REFBIN):
        chk = subprocess.run([REFBIN, "-wcheck", work], capture_output=True, text=True, timeout=600).stdout
        assert "[100.000% OK]" in chk and "Wrong" not in chk, chk[-1500:]


def test_solver_resume_solves(saved):
    work, k, _ = saved
    out = solver(["--resume", work, "--grid", GRID])
    assert "resume: rank 0: %d walks loaded" % NK in out and ", 0 re-created" in out, out[-2000:]
    assert PRIV110 in out, out[-2000:]
    total = int(re.search(r"Total count: (\d+)", out).group(1))
    assert total > (k + 1) * NK * NB_RUN


@pytest.mark.parametrize("grid,fresh", [("64,128", True), ("16,128", False)])
def test_solver_resume_other_grid(saved, grid, fresh):
    work, _, _ = saved
    out = solver(["--resume", work, "--grid", grid])
    if fresh:
        assert "%d created fresh" % (64 * 128 * 128 - NK) in out, out[-2000:]
    else:
        assert "FectchKangaroos: Warning %d unhandled kangaroos" % (NK - 16 * 128 * 128) in out, out[-2000:]
    assert PRIV110 in out, out[-2000:]


def test_solver_rejects_a_file_of_another_key(saved, tmp_path):
    work, _, _ = saved
    raw = bytearray(open(work, "rb").read())
    other = ec.mul(0x35C0D7234DF7DEB0F20CF7062445)                   # a key in the same range, not the saved one
    raw[76:108] = other[0].to_bytes(32, "little"); raw[108:140] = other[1].to_bytes(32, "little")
    bad = str(tmp_path / "other.work")
    open(bad, "wb").write(bytes(raw))
    out = solver(["--resume", bad, "--grid", GRID, "--max-steps", "4"])
    assert "does not belong to this key and range" in out, out[-2000:]


def test_interop_with_the_reference_program(saved, tmp_path):
    if not os.path.exists(DROPIN):
        pytest.skip("oracle/_ref/kangaroo_b200 not built (needs the reference sources at build time)")
    work, _, _ = saved
    out = subprocess.run([DROPIN, "-t", "0", "-gpu", "-g", GRID, "-i", work], capture_output=True, text=True, timeout=900, cwd=ROOT)
    out = out.stdout + out.stderr
    assert "kangaroos loaded" in out and PRIV110 in out.upper(), out[-2000:]
    # a -ws file written by the reference program resumes in the solver
    # -m 0.05: the reference program gives up at 5 % of the expected operations of the 2^72 window (a solve that early has a
    # probability of about 0.2 %) and saves at its first status tick before that (-wi 1, Thread.cpp:326-343)
    ref = str(tmp_path / "ref.work")
    o = subprocess.run([DROPIN, "-t", "0", "-gpu", "-g", GRID, "-d", "10", "-w", ref, "-wi", "1", "-ws", "-m", "0.05",
                        os.path.join(GOLD, "puzzle110_window72.txt")], capture_output=True, text=True, timeout=600, cwd=ROOT)
    if PRIV110 in o.stdout.upper():
        pytest.fail("the reference program solved the key before it gave up: no work file to resume\n" + o.stdout[-2000:])
    assert "Aborted" in o.stdout and os.path.exists(ref), "the reference program wrote no work file\n" + o.stdout[-2000:]
    assert read_work_info(ref).n_walks == NK
    out = solver(["--resume", ref, "--grid", GRID])
    assert ", 0 re-created" in out and PRIV110 in out, out[-2000:]


def test_solver_sigterm_writes_a_checkpoint(tmp_path):
    work = str(tmp_path / "sig.work")
    cfg = os.path.join(GOLD, "puzzle110_window72.txt")
    p = subprocess.Popen([sys.executable, "-m", "kangaroo_b200.solver", cfg, "--dp", "10", "--grid", GRID, "--seed", "9",
                          "--work-file", work, "--save-kangaroos"], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, cwd=ROOT)
    lines = []
    try:
        for line in p.stdout:
            lines.append(line)
            if line.startswith("["):                                 # first status line
                p.send_signal(signal.SIGTERM)
                break
        rest, _ = p.communicate(timeout=300)
    finally:
        if p.poll() is None:
            p.kill()
            p.wait()
    out = "".join(lines) + rest
    assert p.returncode in (0, 1), out[-2000:]
    if "Priv:" in out:
        pytest.fail("the key was found before SIGTERM arrived: pick another seed\n" + out[-2000:])
    assert "checkpoint: " + work in out and read_work_info(work).n_walks == NK, out[-2000:]
    out = solver(["--resume", work, "--grid", GRID])
    assert PRIV110 in out, out[-2000:]


def test_solver_periodic_checkpoints(tmp_path):
    work = str(tmp_path / "per.work")
    out = solver([os.path.join(GOLD, "puzzle110_window80.txt"), "--dp", "10", "--grid", GRID, "--seed", "13", "--max-steps", "1500",
                  "--work-file", work, "--work-interval", "1", "--save-kangaroos"])
    n_ck = out.count("checkpoint: %s  " % work)                     # committed ones
    assert n_ck >= 2, out[-2000:]
    assert "Priv:" not in out                                        # 2^80: out of reach of 1500 steps
    info = read_work_info(work)
    assert info.total_count == 1501 * NK * NB_RUN and info.n_walks == NK


def test_failed_checkpoint_does_not_end_the_run(tmp_path):
    """A checkpoint whose table cannot be written (F.tmp is a directory here) is dropped, the previous F stays, and the run
    goes on: once the obstacle is gone the next checkpoint commits."""
    work = str(tmp_path / "fail.work")
    open(work, "wb").write(b"previous")
    os.mkdir(work + ".tmp")
    p = subprocess.Popen([sys.executable, "-m", "kangaroo_b200.solver", os.path.join(GOLD, "puzzle110_window80.txt"), "--dp", "10",
                          "--grid", GRID, "--seed", "17", "--max-steps", "2500", "--work-file", work, "--work-interval", "1",
                          "--save-kangaroos"], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, cwd=ROOT)
    lines = []
    try:
        for line in p.stdout:
            lines.append(line)
            if "not written, the previous file is kept" in line:
                assert open(work, "rb").read() == b"previous"
                os.rmdir(work + ".tmp")
                break
        rest, _ = p.communicate(timeout=600)
    finally:
        if p.poll() is None:
            p.kill()
            p.wait()
    out = "".join(lines) + rest
    assert p.returncode == 1 and "Key# 0 not found" in out, out[-2000:]
    assert "checkpoint: %s  " % work in out, out[-2000:]
    info = read_work_info(work)
    assert info.total_count == 2501 * NK * NB_RUN and info.n_walks == NK


def test_key_found_while_a_checkpoint_is_written(tmp_path):
    """The default herd (4.85 M walks, 466 MB per checkpoint) with a checkpoint begun at every opportunity: the key of the
    2^64 window arrives while walks are being written.  The run must finish that work before the engine and the table go
    away, drop F.tmp and exit normally."""
    work = str(tmp_path / "race.work")
    p = subprocess.run([sys.executable, "-m", "kangaroo_b200.solver", os.path.join(GOLD, "puzzle110_window64.txt"), "--dp", "8",
                        "--seed", "23", "--work-file", work, "--work-interval", "1e-9", "--save-kangaroos"],
                       capture_output=True, text=True, timeout=900, cwd=ROOT)
    out = p.stdout + p.stderr
    assert p.returncode == 0 and PRIV110 in out, out[-2000:]
    assert "abandoned, the run ended while it was written" in out, out[-2000:]
    assert not os.path.exists(work + ".tmp")


def test_checkpoint_two_gpus_resumes_on_one(tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    work = str(tmp_path / "two.work")
    p = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--standalone", "--nproc-per-node", "2", "-m", "kangaroo_b200.solver",
                        os.path.join(GOLD, "puzzle110_window64.txt"), "--dp", "10", "--grid", GRID, "--seed", "3", "--max-steps", "6",
                        "--work-file", work, "--save-kangaroos"], capture_output=True, text=True, timeout=900, cwd=ROOT)
    out = p.stdout + p.stderr
    assert PRIV110 not in out, "solved before the checkpoint\n" + out[-2000:]
    assert read_work_info(work).n_walks == 2 * NK, out[-2000:]
    out = solver(["--resume", work, "--grid", "64,128"])
    assert "%d walks loaded" % (2 * NK) in out and "0 created fresh" in out and PRIV110 in out, out[-2000:]
