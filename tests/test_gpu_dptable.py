"""-m gpu: the device DP table (kgx_dpt_*, kangaroo_b200/dptable.py) against the host table (kgx_ingest.cpp), and the solver
on it (KGX_DPTABLE=device): solves, checkpoints, resume across table kinds, SIGTERM, migration to the host table."""
import os
import re
import signal
import subprocess
import sys

import numpy as np
import pytest

from kangaroo_b200.dptable import DeviceDPTable
from kangaroo_b200.ingest import DPTable, read_work_info

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")
REFBIN = os.path.join(ROOT, "oracle", "_ref", "kangaroo_ref_cpu")
PRIV110 = "35C0D7234DF7DEB0F20CF7062444"
GRID = "32,128"
DP40 = np.dtype([("kidx", "<u4"), ("h", "<u4"), ("x", "<u8", 2), ("d", "<u8", 2)])
TYPE = np.uint64(1 << 62)
KEY = (0x79BE667EF9DCBBAC55A06295CE870B07029BFCDB2DCE28D959F2815B16F81798,
       0x483ADA7726A3C4655DA4FBFC0E1108A8FD17B448A68554199C47D08FFB10D4B8)


def _torch():
    import torch
    return torch


def _records(rng, n, buckets):
    r = np.zeros(n, dtype=DP40)
    r["kidx"] = rng.integers(0, 1 << 20, n)
    r["h"] = rng.integers(0, buckets, n)
    r["x"] = rng.integers(0, 1 << 63, (n, 2), dtype=np.uint64)
    r["d"] = rng.integers(0, 1 << 62, (n, 2), dtype=np.uint64)
    return r


def _variants(rng, src, k):
    """k records re-using keys of src: exact duplicates, same-herd and tame/wild collisions (other d, type kept / flipped)"""
    out = src[rng.integers(0, len(src), k)].copy()
    kind = rng.integers(0, 3, k)
    out["d"][kind >= 1, 0] += np.uint64(1)
    out["d"][kind == 2, 1] ^= TYPE
    out["kidx"] = rng.integers(0, 1 << 20, k)
    return out


def _streams(seed=1, world=3, steps=6, per=4000, buckets=1 << 18):
    """steps x world batches with every kind of repeat, across and inside batches"""
    rng = np.random.default_rng(seed)
    seen, steps_out = _records(rng, 1, buckets), []
    for _ in range(steps):
        batch = []
        for _r in range(world):
            fresh = _records(rng, per, buckets)
            inside = _variants(rng, fresh, per // 20)                # repeats of this batch's own records
            older = _variants(rng, seen, per // 20)                  # repeats of earlier batches
            recs = np.concatenate([fresh, inside, older])
            batch.append(recs[rng.permutation(len(recs))])
        seen = np.concatenate([seen] + batch)
        steps_out.append(batch)
    return steps_out


def _flat(torch, batch):
    """one device buffer, rank r at r * cap records (the layout of DPGather.step_flat)"""
    cap = max(len(b) for b in batch) + 17
    buf = np.zeros(len(batch) * cap, dtype=DP40)
    for r, b in enumerate(batch):
        buf[r * cap: r * cap + len(b)] = b
    return torch.from_numpy(buf.view(np.uint8).copy()).cuda(), cap


def _feed(torch, steps, dev, host):
    ev_d, ev_h = [], []
    for batch in steps:
        flat, cap = _flat(torch, batch)
        dev.insert(flat.data_ptr(), [len(b) for b in batch], cap, torch.cuda.current_stream().cuda_stream)
        for r, b in enumerate(batch):
            ev_h += host.add_dp40(b.view(np.uint8), r)
        if dev.pending == 2:
            ev_d += dev.events()
        torch.cuda.synchronize()                                    # flat is freed at the next iteration
    while dev.pending:
        ev_d += dev.events()
    return ev_d, ev_h


def _file(table, path):
    table.save_work(str(path), 10, 1 << 40, (1 << 41) - 1, KEY, total_count=5, total_time=1.0)
    return open(path, "rb").read()


def _normalised(host, path):
    """the host table's content written the way a device export is: kgi_export_sorted -> kgi_fill_sorted"""
    h, e = host.export_sorted()
    t = DPTable(threads=1)
    t.fill_sorted(h, e)
    b = _file(t, path)
    t.close()
    return b


def test_device_table_matches_host_table(tmp_path):
    torch = _torch()
    steps = _streams()
    dev, host = DeviceDPTable(0, 1 << 20), DPTable(threads=4)
    ev_d, ev_h = _feed(torch, steps, dev, host)
    kinds = {k for k, *_ in ev_h}
    assert kinds == {1, 2} and len(ev_h) > 1000
    assert sorted(ev_d) == sorted(ev_h)
    assert dev.count() == len(host) == dev.entries
    out = DPTable(threads=1)
    dev.to_host(out)
    assert _file(out, tmp_path / "d.work") == _normalised(host, tmp_path / "h.work")
    # a record with h >= 2^18 is refused by both, the rest of its batch is inserted
    bad = _records(np.random.default_rng(9), 50, 1 << 18)
    bad["h"][7] = 1 << 18
    flat, cap = _flat(torch, [bad])
    dev.insert(flat.data_ptr(), [len(bad)], cap, torch.cuda.current_stream().cuda_stream)
    with pytest.raises(RuntimeError, match="h >= 2"):
        dev.events()
    with pytest.raises(RuntimeError, match="h >= 2"):
        host.add_dp40(bad.view(np.uint8))
    assert dev.count() == len(host)
    dev.to_host(out)
    assert _file(out, tmp_path / "d2.work") == _normalised(host, tmp_path / "h2.work")
    dev.close(); host.close(); out.close()


def test_crowded_buckets_and_chunked_export(tmp_path):
    """few buckets: long probe runs across bucket borders, exports split inside the bucket range"""
    torch = _torch()
    steps = _streams(seed=4, world=2, steps=4, per=20000, buckets=64)
    dev, host = DeviceDPTable(0, 1 << 20), DPTable(threads=2)
    ev_d, ev_h = _feed(torch, steps, dev, host)
    assert sorted(ev_d) == sorted(ev_h)
    out = DPTable(threads=1)
    dev.export_begin()
    out.reset()
    for h, e in dev.export_chunks(chunk=9000):                      # several buckets per chunk, never a split bucket
        out.fill_sorted(h, e)
    dev.export_end()
    assert _file(out, tmp_path / "d.work") == _normalised(host, tmp_path / "h.work")
    dev.close(); host.close(); out.close()


def test_export_is_a_snapshot(tmp_path):
    """an export begun after insert L holds inserts 1..L, even when later inserts run before it is read"""
    torch = _torch()
    steps = _streams(seed=6, world=1, steps=4, per=30000)
    dev, host = DeviceDPTable(0, 1 << 20), DPTable(threads=2)
    _feed(torch, steps[:2], dev, host)
    stream = torch.cuda.current_stream().cuda_stream
    dev.export_begin(stream)
    for batch in steps[2:]:
        flat, cap = _flat(torch, batch)
        dev.insert(flat.data_ptr(), [len(b) for b in batch], cap, stream)
        torch.cuda.synchronize()
        dev.events()
    out = DPTable(threads=1)
    dev.export_to_host(out)
    assert _file(out, tmp_path / "d.work") == _normalised(host, tmp_path / "h.work")
    dev.close(); host.close(); out.close()


def test_engine_dps_match():
    """real DPs of several launches (dp 8, small grid) through both tables"""
    torch = _torch()
    from kangaroo_b200 import GPUEngine, random_herd_arrays
    from kangaroo_b200 import ecmath as ec
    from kangaroo_b200.dist import SlabView
    from kangaroo_b200.solver import create_jump_table, dp_mask
    eng = GPUEngine(8, 128, 0, 1 << 17)                               # about 32 k DPs per launch, below max_found
    eng.SetParams(dp_mask(8), *create_jump_table(64))
    eng.SetWildOffset(1 << 63)
    sc, d128 = random_herd_arrays(eng.nbKangaroo, 64, 1 << 63, np.random.Generator(np.random.PCG64(3)))
    eng.CreateHerdRaw(sc, d128, ec.mul(0x1234567))
    dev, host = DeviceDPTable(0, 1 << 20), DPTable(threads=4)
    ev_d, ev_h, total = [], [], 0
    eng.callKernel()
    for _ in range(6):
        n = min(eng.collect_count(relaunch=True), eng.maxFound)
        assert n > 0
        ptr = eng.convert_dps_device_ptr()
        recs = torch.as_tensor(SlabView(ptr + 4, n * 40), device="cuda").clone()
        total += n
        dev.insert(recs.data_ptr(), [n])
        ev_h += host.add_dp40(recs.cpu().numpy())
        ev_d += dev.events()
    eng.sync()
    assert total > 10000
    assert sorted(ev_d) == sorted(ev_h) and dev.count() == len(host)
    out = DPTable(threads=1)
    dev.to_host(out)
    h1, e1 = out.export_sorted()
    h2, e2 = host.export_sorted()
    assert np.array_equal(h1, h2) and np.array_equal(e1, e2)
    eng.close(); dev.close(); host.close(); out.close()


def test_save_load_export_round_trip(tmp_path):
    rng = np.random.default_rng(8)
    recs = _records(rng, 200000, 1 << 18)
    host = DPTable(threads=4)
    host.add_dp40(recs.view(np.uint8))
    src = _normalised(host, tmp_path / "src.work")
    loaded = DPTable(threads=1)
    read_work_info(str(tmp_path / "src.work"), loaded)
    dev = DeviceDPTable(0, 1 << 20)
    dev.load_from_host(loaded)
    assert dev.count() == len(recs)
    out = DPTable(threads=1)
    dev.to_host(out)
    assert _file(out, tmp_path / "again.work") == src
    for t in (host, loaded, out):
        t.close()
    dev.close()


# ---- the solver on the device table -----------------------------------------------------------------------------------
def solver(args, env=None, timeout=900):
    e = dict(os.environ, KGX_DPTABLE="device")
    e.update(env or {})
    p = subprocess.run([sys.executable, "-m", "kangaroo_b200.solver"] + args, capture_output=True, text=True, timeout=timeout,
                       cwd=ROOT, env=e)
    return p.stdout + p.stderr


def test_solver_in56_device():
    out = solver([os.path.join(GOLD, "in56.txt"), "--dp", "8", "--grid", GRID, "--seed", "7"])
    assert "DP table: device" in out and "Suggested DP:" in out and "Expected operations: 2^" in out, out[-2000:]
    assert "Priv: 0x3447F65ABC9F46F736A95F87B044829C8A0129D56782D635CD612C0F05F3DA03" in out, out[-2000:]


def test_solver_puzzle110_window_device():
    out = solver([os.path.join(GOLD, "puzzle110_window56.txt"), "--dp", "8", "--grid", GRID, "--seed", "11"])
    assert "DP table: device" in out and "Priv: 0x" + PRIV110 in out, out[-2000:]


def test_default_choice_is_the_device_table_on_small_runs():
    out = solver([os.path.join(GOLD, "puzzle110_window56.txt"), "--dp", "8", "--grid", GRID, "--seed", "11"], env={"KGX_DPTABLE": "auto"})
    assert "DP table: device" in out and "Priv: 0x" + PRIV110 in out, out[-2000:]


def _table_of(path):
    t = DPTable(threads=1)
    read_work_info(path, t)
    r = t.export_sorted()
    t.close()
    return r


def test_migration_ends_with_the_host_tables_content(tmp_path):
    """the solver's migration: a device table that would overflow hands its content to the host table (export ->
    kgi_fill_sorted) and the records go on there; events and content match a host table fed from the start"""
    torch = _torch()
    steps = _streams(seed=12, world=2, steps=6, per=5000)
    dev, mig, host = DeviceDPTable(0, 25000), DPTable(threads=2), DPTable(threads=2)
    ev_m, ev_h, moved = [], [], False
    for batch in steps:
        n = sum(len(b) for b in batch)
        for r, b in enumerate(batch):
            ev_h += host.add_dp40(b.view(np.uint8), r)
        if dev is not None:
            while dev.pending:
                ev_m += dev.events()
            if dev.fits(n):
                flat, cap = _flat(torch, batch)
                dev.insert(flat.data_ptr(), [len(b) for b in batch], cap, torch.cuda.current_stream().cuda_stream)
                ev_m += dev.events()
                continue
            dev.to_host(mig)
            dev.close()
            dev, moved = None, True
        for r, b in enumerate(batch):
            ev_m += mig.add_dp40(b.view(np.uint8), r)
    assert moved and sorted(ev_m) == sorted(ev_h) and len(mig) == len(host)
    assert _normalised(mig, tmp_path / "m.work") == _normalised(host, tmp_path / "h.work")
    mig.close(); host.close()


@pytest.mark.parametrize("cap", [None, "200000"])
def test_solver_save_work_device(tmp_path, cap):
    """--save-work from the device table, also after a migration mid-run: the file holds every DP the run reports"""
    work = str(tmp_path / "d.work")
    env = {"KGX_DPTABLE_CAP": cap} if cap else {}
    out = solver([os.path.join(GOLD, "puzzle110_window80.txt"), "--dp", "8", "--grid", GRID, "--seed", "31", "--max-steps", "10",
                  "--save-work", work], env=env)
    assert "DP table: device" in out and ("device table is full" in out) == bool(cap), out[-2000:]
    n = int(re.search(r"; (\d+) DPs;", out).group(1))
    assert n > 200000 and len(_table_of(work)[0]) == n, out[-2000:]


def test_forced_migration_still_solves():
    out = solver([os.path.join(GOLD, "puzzle110_window56.txt"), "--dp", "8", "--grid", GRID, "--seed", "11"],
                 env={"KGX_DPTABLE_CAP": "30000"})
    assert "device table is full" in out and "Priv: 0x" + PRIV110 in out, out[-2000:]


@pytest.fixture(scope="module")
def saved_dev(tmp_path_factory):
    work = str(tmp_path_factory.mktemp("ckd") / "p110.work")
    out = solver([os.path.join(GOLD, "puzzle110_window64.txt"), "--dp", "10", "--grid", GRID, "--seed", "5", "--max-steps", "12",
                  "--work-file", work, "--save-kangaroos"])
    assert PRIV110 not in out and "checkpoint: " + work in out and "DP table: device" in out, out[-2000:]
    return work


def test_device_checkpoint_file(saved_dev):
    info = read_work_info(saved_dev)
    assert info.n_walks == 32 * 128 * 128 and os.path.getsize(saved_dev) == info.walk_offset + 96 * info.n_walks
    if os.path.exists(REFBIN):
        chk = subprocess.run([REFBIN, "-wcheck", saved_dev], capture_output=True, text=True, timeout=600).stdout
        assert "[100.000% OK]" in chk and "Wrong" not in chk, chk[-1500:]


@pytest.mark.parametrize("kind", ["device", "host"])
def test_resume_device_checkpoint(saved_dev, kind):
    out = solver(["--resume", saved_dev, "--grid", GRID], env={"KGX_DPTABLE": kind})
    assert "DP table: " + kind in out and ", 0 re-created" in out and PRIV110 in out, out[-2000:]


def test_resume_host_checkpoint_on_device(tmp_path):
    work = str(tmp_path / "h.work")
    out = solver([os.path.join(GOLD, "puzzle110_window64.txt"), "--dp", "10", "--grid", GRID, "--seed", "5", "--max-steps", "12",
                  "--work-file", work, "--save-kangaroos"], env={"KGX_DPTABLE": "host"})
    assert "DP table: host" in out and "checkpoint: " + work in out, out[-2000:]
    n = len(_table_of(work)[0])
    out = solver(["--resume", work, "--grid", GRID, "--max-steps", "1"])
    assert "DP table: device" in out, out[-2000:]
    assert int(re.search(r"; (\d+) DPs;", out).group(1)) >= n, out[-2000:]
    out = solver(["--resume", work, "--grid", GRID])
    assert PRIV110 in out, out[-2000:]


def test_sigterm_writes_a_device_checkpoint(tmp_path):
    work = str(tmp_path / "sig.work")
    env = dict(os.environ, KGX_DPTABLE="device")
    p = subprocess.Popen([sys.executable, "-m", "kangaroo_b200.solver", os.path.join(GOLD, "puzzle110_window72.txt"), "--dp", "10",
                          "--grid", GRID, "--seed", "9", "--work-file", work, "--save-kangaroos"], stdout=subprocess.PIPE,
                         stderr=subprocess.STDOUT, text=True, cwd=ROOT, env=env)
    lines = []
    try:
        for line in p.stdout:
            lines.append(line)
            if line.startswith("["):
                p.send_signal(signal.SIGTERM)
                break
        rest, _ = p.communicate(timeout=300)
    finally:
        if p.poll() is None:
            p.kill()
            p.wait()
    out = "".join(lines) + rest
    if "Priv:" in out:
        pytest.fail("the key was found before SIGTERM arrived: pick another seed\n" + out[-2000:])
    assert "DP table: device" in out and "checkpoint: " + work in out, out[-2000:]
    assert read_work_info(work).n_walks == 32 * 128 * 128
    out = solver(["--resume", work, "--grid", GRID])
    assert PRIV110 in out, out[-2000:]


def test_two_gpus_device_table(tmp_path):
    torch = _torch()
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    env = dict(os.environ, KGX_DPTABLE="device")
    p = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--standalone", "--nproc-per-node", "2", "-m", "kangaroo_b200.solver",
                        os.path.join(GOLD, "puzzle110_window56.txt"), "--dp", "8", "--grid", GRID, "--seed", "3"],
                       capture_output=True, text=True, timeout=900, cwd=ROOT, env=env)
    out = p.stdout + p.stderr
    assert "DP table: device" in out and PRIV110 in out, out[-2000:]
