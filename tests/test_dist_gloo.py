"""world_size-2 gloo test (CPU) of the DP gather logic used for the multi-GPU path (kangaroo_b200/dist.py)."""
import os
import socket
import struct

import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from kangaroo_b200.dist import DPGather, decode_records, ITEM_BYTES


def _records(rank, n):
    out = b""
    for i in range(n):
        x = (rank << 200) | (i * 0x1234567 + 1)
        d = (rank << 100) | i
        out += x.to_bytes(32, "little") + d.to_bytes(16, "little") + struct.pack("<Q", rank * 1000 + i)
    return out


def _worker(rank, world, port, q):
    os.environ["MASTER_ADDR"] = "127.0.0.1"; os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    max_found = 1024
    results = []
    for step, counts in enumerate([(3, 700), (0, 0), (1024, 5), (300, 300)]):
        n = counts[rank]
        slab = torch.zeros(4 + max_found * ITEM_BYTES, dtype=torch.uint8)
        raw = struct.pack("<I", n) + _records(rank, n)
        slab[:len(raw)] = torch.frombuffer(bytearray(raw), dtype=torch.uint8)
        g = DPGather(None, dist, rank, world, torch, device=torch.device("cpu"), slab_fn=lambda s=slab: s, max_found=max_found)
        out = g.step(n)
        if rank == 0:
            got = {r: decode_records(buf) for r, buf in out}
            results.append({r: len(v) for r, v in got.items()})
            for r in range(world):
                exp = decode_records(_records(r, counts[r]))
                assert got[r] == exp, (step, r)
        else:
            assert out is None
    if rank == 0:
        q.put(results)
    dist.destroy_process_group()


def test_dp_gather_world2_gloo():
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = q.get(timeout=120)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    assert res == [{0: 3, 1: 700}, {0: 0, 1: 0}, {0: 1024, 1: 5}, {0: 300, 1: 300}]


# ---- the solver's data plane: 40-byte DP records -> step_flat gather -> rank-0 reference HashTable (ingest.DPTable) --------
def _dp40(rank, n, dup_of_rank0=0):
    """n distinct records of `rank` (x unique per (rank, i)); the first dup_of_rank0 repeat rank 0's records exactly."""
    out = b""
    for i in range(n):
        src = 0 if i < dup_of_rank0 else rank
        x = ((src + 1) << 100) | (i * 0x9E3779B97F4A7C15 & ((1 << 90) - 1))
        d = ((src + 7) << 64) | i | ((i & 1) << 126)
        h = (i * 2654435761 + src) & 0x3FFFF
        out += struct.pack("<IIQQQQ", rank * 100000 + i, h, x & (2**64 - 1), x >> 64, d & (2**64 - 1), d >> 64)
    return out


def _worker_flat(rank, world, port, q):
    import numpy as np
    os.environ["MASTER_ADDR"] = "127.0.0.1"; os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from kangaroo_b200.dist import DP40_BYTES
    max_found = 2048
    table = None
    if rank == 0:
        from kangaroo_b200.ingest import DPTable, EV_RESET
        table = DPTable(threads=2)
    log = []
    for step, counts in enumerate([(500, 1500), (0, 40), (2048, 1)]):
        n = counts[rank]
        recs = _dp40(rank, n, dup_of_rank0=(25 if (rank == 1 and step == 0) else 0))
        slab = torch.zeros(4 + max_found * DP40_BYTES, dtype=torch.uint8)
        raw = struct.pack("<I", n) + recs
        slab[:len(raw)] = torch.frombuffer(bytearray(raw), dtype=torch.uint8)
        g = DPGather(None, dist, rank, world, torch, device=torch.device("cpu"), slab_fn=lambda s=slab: s, max_found=max_found, wire="dp40")
        res = g.step_flat(n)
        if rank == 0:
            cnts, cap, flat = res
            assert cnts == list(counts)
            h = flat.numpy()
            events = []
            for r in range(world):
                seg = h[r * cap * DP40_BYTES: r * cap * DP40_BYTES + cnts[r] * DP40_BYTES]
                assert bytes(seg) == _dp40(r, cnts[r], dup_of_rank0=(25 if (r == 1 and step == 0) else 0))
                events += table.add_dp40(np.ascontiguousarray(seg), r)
            log.append((len(table), sorted((e[1], e[2]) for e in events if e[0] == EV_RESET)))
        else:
            assert res is None
    if rank == 0:
        q.put(log)
        table.close()
    dist.destroy_process_group()


def test_flat_gather_into_reference_hashtable_world2_gloo():
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker_flat, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    log = q.get(timeout=120)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    # step 0: 500 + 1500 records, 25 of rank 1's are exact copies of rank 0's -> 25 reset requests tagged (rank 1, its kIdx)
    assert log[0] == (500 + 1500 - 25, [(1, 100000 + i) for i in range(25)])
    # step 1: rank 1 re-sends its first 40 own records: 25 of them are new (step 0 carried rank 0's copies instead), 15 duplicates
    assert log[1] == (2000, [(1, 100000 + i) for i in range(25, 40)])
    # step 2: rank 0 sends 2048 (first 500 stored already), rank 1 one stored record
    assert log[2][0] == 2000 + (2048 - 500) and len(log[2][1]) == 500 + 1
