"""CPU: work files that carry kangaroos (kgi_save_work_walks / kgi_load_work_ex in kangaroo_b200/csrc/kgx_ingest.cpp), the
walk-record convention of the reference's -ws files, and the multi-writer checkpoint protocol (kangaroo_b200/checkpoint.py)."""
import gzip
import os
import socket
import struct

import numpy as np
import pytest

from kangaroo_b200 import checkpoint as ckpt
from kangaroo_b200 import ecmath as ec
from kangaroo_b200.ingest import DPTable, read_work_info
from oracle import kgo

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HASH_SIZE = 1 << 18
M64 = (1 << 64) - 1
START = 0x5B3F38AF935A3640D158E871CE6E9666DB862636383386EE0000000000000000
END = START + (1 << 64) - 1
PUB = ec.mul(START + 0x18CCC3BD72EB)


def _filled_table(n=3000, seed=5):
    rng = np.random.default_rng(seed)
    raw = np.zeros((n, 10), dtype=np.uint32)
    raw[:, 0] = np.arange(n)
    raw[:, 2:10] = rng.integers(0, 1 << 32, size=(n, 8), dtype=np.uint32)
    raw[:, 1] = raw[:, 6] & 0x3FFFF
    raw[:, 9] &= 0x3FFFFFFF
    t = DPTable(threads=2)
    t.add_dp40(raw)
    assert len(t) == n
    return t


def test_save_work_walks_layout(tmp_path):
    t = _filled_table()
    plain, walks = str(tmp_path / "plain.work"), str(tmp_path / "walks.work")
    t.save_work(plain, 14, START, END, PUB, total_count=123456789, total_time=42.5)
    nw = 4096
    off = t.save_work_walks(walks, 14, START, END, PUB, total_count=123456789, total_time=42.5, total_walks=nw)
    a, b = open(plain, "rb").read(), open(walks, "rb").read()
    assert off == 156 + HASH_SIZE * 8 + 32 * len(t) + 8 == len(a)
    assert len(b) == off + 96 * nw
    assert b[:off - 8] == a[:-8]                                   # same header and table
    assert struct.unpack("<Q", a[-8:])[0] == 0 and struct.unpack("<Q", b[off - 8:off])[0] == nw
    assert b[off:] == bytes(96 * nw)                               # room for the walks, not yet written
    t.close()


def test_load_work_ex_round_trip(tmp_path):
    t = _filled_table(n=777)
    path = str(tmp_path / "w.work")
    off = t.save_work_walks(path, 9, START, END, PUB, total_count=(1 << 50) + 3, total_time=1.25e5, total_walks=10)
    for table in (None, DPTable(threads=1)):
        info = read_work_info(path, table)
        assert (info.dp_bits, info.range_start, info.range_end, info.key) == (9, START, END, PUB)
        assert (info.total_count, info.total_time, info.n_walks, info.walk_offset) == ((1 << 50) + 3, 1.25e5, 10, off)
        if table is not None:
            assert len(table) == 777
            table.close()
    # a key off the curve is refused (Backup.cpp:175-179)
    raw = bytearray(open(path, "rb").read())
    raw[12 + 64 + 32] ^= 1                                        # one bit of key.y
    bad = str(tmp_path / "bad.work")
    open(bad, "wb").write(bytes(raw))
    with pytest.raises(ValueError, match="curve"):
        read_work_info(bad)
    open(bad, "wb").write(b"not a work file")
    with pytest.raises(RuntimeError):
        read_work_info(bad)
    t.close()


def test_reference_ws_file_walk_convention(oracle, tmp_path):
    """A work file the reference's CPU program wrote with -ws (tests/golden/make_ref_walks.py): every record i is
    {x, y, d} with d*G = (x, y) for even i (tame) and key + d*G = (x, y) for odd i (wild), key = P - start*G, d mod n --
    negative wild distances included."""
    path = str(tmp_path / "ref.work")
    with gzip.open(os.path.join(ROOT, "tests", "golden", "ref_walks_in80.work.gz"), "rb") as g:
        open(path, "wb").write(g.read())
    info = read_work_info(path)
    assert info.n_walks == 2048 and info.dp_bits == 20
    assert os.path.getsize(path) == info.walk_offset + 96 * info.n_walks
    start, end, pubs = ec.parse_config(os.path.join(ROOT, "tests", "golden", "in80.txt"))
    assert (info.range_start, info.range_end, info.key) == (start, end, pubs[0])
    key = ec.add(info.key, ec.neg(ec.mul(info.range_start)))
    recs = np.fromfile(path, dtype=np.uint64, offset=info.walk_offset).reshape(-1, 12)
    neg = 0
    for i, r in enumerate(recs):
        x, y, d = kgo.from_limbs(r[0:4]), kgo.from_limbs(r[4:8]), kgo.from_limbs(r[8:12])
        assert d < kgo.N
        p = oracle.ec_mul_g(d)
        if i & 1:
            p = oracle.ec_add(key, p)
            neg += d > kgo.N // 2
        assert p == (x, y), i
    assert neg > 0                                               # some wild walks are still below the range's middle


# ---- the multi-writer protocol under gloo ------------------------------------------------------------------------------
N_PER_RANK = 1000


def _walks(rank, n):
    rng = np.random.default_rng(100 + rank)
    return rng.integers(0, 1 << 63, size=(n, 12), dtype=np.uint64)


def _ck_worker(rank, world, port, path, fail_rank, q):
    import torch
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"; os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        flag = torch.zeros(1, dtype=torch.int64)
        if rank == 0:                                              # header + table, file at its final size
            t = _filled_table(n=500)
            flag[0] = t.save_work_walks(ckpt.tmp_path(path), 12, START, END, PUB, 99, 1.5, world * N_PER_RANK)
            t.close()
        dist.broadcast(flag, 0)
        offset = int(flag.item())
        mine = _walks(rank, N_PER_RANK)
        buf = np.empty(7 * 12, dtype=np.uint64)                   # 7-walk chunks: slices end mid-chunk

        def read(b, first, count):
            if rank == fail_rank and first >= 500:
                raise OSError("simulated write failure")
            b[:count * 12] = mine[first:first + count].reshape(-1)
        w = ckpt.SliceWriter(ckpt.tmp_path(path), offset, rank * N_PER_RANK, N_PER_RANK, read, buf, 7)
        w.join()
        flag[0] = w.state
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        if rank == 0:
            if int(flag.item()) == 1:
                ckpt.commit(path)
            else:
                ckpt.discard(path)
            q.put(int(flag.item()))
    finally:
        dist.destroy_process_group()


def _run_world2(path, fail_rank):
    import torch.multiprocessing as mp
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_ck_worker, args=(r, 2, port, path, fail_rank, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = q.get(timeout=120)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    return res


def test_slice_writers_world2_equal_single_writer(tmp_path):
    path = str(tmp_path / "ck.work")
    assert _run_world2(path, fail_rank=-1) == 1
    assert not os.path.exists(ckpt.tmp_path(path))
    single = str(tmp_path / "single.work")
    t = _filled_table(n=500)
    off = t.save_work_walks(single, 12, START, END, PUB, 99, 1.5, 2 * N_PER_RANK)
    t.close()
    with open(single, "r+b") as f:
        f.seek(off)
        for r in range(2):
            f.write(_walks(r, N_PER_RANK).tobytes())
    assert open(path, "rb").read() == open(single, "rb").read()


def test_failed_writer_keeps_previous_file(tmp_path):
    path = str(tmp_path / "ck.work")
    open(path, "wb").write(b"previous checkpoint")
    assert _run_world2(path, fail_rank=1) == -1
    assert open(path, "rb").read() == b"previous checkpoint"
    assert not os.path.exists(ckpt.tmp_path(path))
