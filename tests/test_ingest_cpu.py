"""CPU: the rank-0 DP ingest (kangaroo_b200/csrc/libkgx_ingest.so = kgx_ingest.cpp).
Semantics pinned to Kangaroo::AddToTable / CollisionCheck / CheckKey (Kangaroo.cpp:218-330), and the work file written by
kgi_save_work to the one the reference's HashTable writes for the same records (tests/golden/work_file_golden.json), plus the
reference's own work-file checker (`kangaroo -wcheck`, Check.cpp:33-108,290-411) where oracle/_ref is built."""
import hashlib
import json
import os
import struct
import subprocess
import time

import numpy as np

from kangaroo_b200 import ecmath as ec
from kangaroo_b200.ingest import LIB_PATH as INGEST
from oracle import kgo

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REFBIN = os.path.join(ROOT, "oracle", "_ref", "kangaroo_ref_cpu")

M64 = (1 << 64) - 1


def rec40(oracle, x, d, ktype, kidx):
    h, X, D = oracle.hash_convert(x, d % kgo.N, ktype)
    return struct.pack("<IIQQQQ", kidx & 0xFFFFFFFF, h, X & M64, X >> 64, D & M64, D >> 64)


def test_exports_every_declared_symbol():
    import ctypes
    import re
    from kangaroo_b200 import ingest
    lib = ctypes.CDLL(INGEST)
    hdr = open(os.path.join(ROOT, "include", "kgx_ingest.h")).read()
    declared = sorted(set(re.findall(r"\b(kgi_[a-z_0-9]+)\s*\(", hdr)))
    assert declared == ingest.EXPORTED_SYMBOLS
    for name in declared:
        getattr(lib, name)


def test_add_semantics_match_add_to_table(oracle):
    from kangaroo_b200.ingest import DPTable, EV_RESET, EV_COLLISION
    rng = np.random.default_rng(7)
    t = DPTable(threads=3, max_events=8192)
    n = 5000
    xs = [int.from_bytes(rng.bytes(32), "little") for _ in range(n)]
    ds = [int.from_bytes(rng.bytes(15), "little") for _ in range(n)]
    buf = b"".join(rec40(oracle, xs[i], ds[i], i & 1, i) for i in range(n))
    assert t.add_dp40(buf, rank=0) == [] and len(t) == n
    # the same records again: ADD_DUPLICATE for every one -> AddToTable false -> reset requests (Kangaroo.cpp:600-609)
    ev = t.add_dp40(buf, rank=3)
    assert len(ev) == n and all(e[0] == EV_RESET and e[1] == 3 for e in ev) and sorted(e[2] for e in ev) == list(range(n))
    assert len(t) == n
    # same x, other distance, same herd -> reset; other herd -> collision carrying both tagged distances
    same = rec40(oracle, xs[10], ds[10] + 5, 10 & 1, 777)
    other = rec40(oracle, xs[11], ds[11] + 9, (11 & 1) ^ 1, 888)
    ev = t.add_dp40(same + other, rank=1)
    kinds = {e[2]: e for e in ev}
    assert kinds[777][0] == EV_RESET and kinds[888][0] == EV_COLLISION
    _, _, Dold = oracle.hash_convert(xs[11], ds[11], 11 & 1)
    _, _, Dnew = oracle.hash_convert(xs[11], ds[11] + 9, (11 & 1) ^ 1)
    assert kinds[888][3] == (Dold & M64, Dold >> 64) and kinds[888][4] == (Dnew & M64, Dnew >> 64)
    # negative wild distances (mod n) keep sign|type tagging through the same path
    neg = rec40(oracle, xs[12] ^ 1, kgo.N - 12345, 1, 5)
    assert t.add_dp40(neg) == [] and len(t) == n + 1
    t.close()


def test_items56_path_equals_device_convert_path(oracle):
    """kgi_add_items (host HashTable::Convert on raw engine ITEMs, biased distances) builds the same table as kgi_add on
    40-byte records."""
    from kangaroo_b200.ingest import DPTable
    rng = np.random.default_rng(11)
    wo = (1 << 79) - 1
    n = 3000
    a, b = DPTable(threads=2, max_events=8192), DPTable(threads=1, max_events=8192)
    items, recs = [], []
    for i in range(n):
        x = int.from_bytes(rng.bytes(32), "little")
        dist = int.from_bytes(rng.bytes(10), "little")                  # true distance; wild ones may be negative
        ktype = i & 1
        true_d = (dist - wo) % kgo.N if ktype else dist
        biased = (true_d + wo) % kgo.N if ktype else true_d               # GPUEngine.cu:407-411
        items.append(struct.pack("<QQQQQQQ", *[(x >> (64 * k)) & M64 for k in range(4)], biased & M64, (biased >> 64) & M64, i))
        recs.append(rec40(oracle, x, true_d, ktype, i))
    assert a.add_items(b"".join(items), wo) == [] and b.add_dp40(b"".join(recs)) == []
    assert len(a) == len(b) == n
    # cross-insert: every record must now be a duplicate in the other table (same h, x, tagged d)
    assert len(a.add_dp40(b"".join(recs))) == n and len(b.add_items(b"".join(items), wo)) == n
    a.close(); b.close()


def test_collision_resolves_to_the_key(oracle):
    """Kangaroo::CollisionCheck -> CheckKey (Kangaroo.cpp:218-302) with the reference's Secp256K1, incl. the symmetric hit."""
    from kangaroo_b200.ingest import DPTable, EV_COLLISION
    start = 0x5B3F38AF935A3640D158E871CE6E9666DB862636383386EE0000000000000000
    priv = start + 0x123456789ABCDEF0
    pub = ec.mul(priv)
    key = ec.add(pub, ec.neg(ec.mul(start)))                              # Kangaroo::InitSearchKey (:892-909)
    t = DPTable(threads=2)
    dt = 0x7777777777777777
    for sym in (False, True):
        # tame at dt*G, wild at key + dw*G = the same point (or, sym, its negative: same x)
        dw = (dt - (priv - start)) % kgo.N if not sym else (-dt - (priv - start)) % kgo.N
        x = ec.mul(dt)[0]
        assert ec.add(key, ec.mul(dw))[0] == x
        t.reset()
        assert t.add_dp40(rec40(oracle, x, dt, 0, 2)) == []
        ev = t.add_dp40(rec40(oracle, x, dw, 1, 3))
        assert len(ev) == 1 and ev[0][0] == EV_COLLISION
        assert t.resolve(ev[0][3], ev[0][4], key, start) == priv
        # same herd twice is never a solution
        assert t.resolve(ev[0][3], ev[0][3], key, start) is None
    t.close()


def test_work_file_passes_the_reference_wcheck(oracle, tmp_path):
    """f3 format half: DPs of a real walk -> kgi_add_items -> kgi_save_work.  The file must be byte for byte the one the
    reference's HashTable::SaveTable writes for the same records (tests/golden/work_file_golden.json);
    where the reference build exists, its own `-winfo` reads the header and `-wcheck` recomputes d*G (+P) for every stored DP
    and compares x and the bucket (Check.cpp:33-108)."""
    from kangaroo_b200.ingest import DPTable
    rp = 64
    start = 0x5B3F38AF935A3640D158E871CE6E9666DB862636383386EE0000000000000000
    end = start + (1 << rp) - 1
    priv = start + 0x18CCC3BD72EB
    pub = ec.mul(priv)
    key = ec.add(pub, ec.neg(ec.mul(start)))
    table = oracle.create_jump_table(rp)
    wdiv2 = ((1 << rp) - 1) >> 1
    oracle.rseed(99)
    px, py, d = oracle.create_herd(2048, rp, wdiv2, key, 0)
    dps = oracle.jump_cpu(px, py, d, table, 256, oracle.dp_mask(6), grp=1024, max_dp=1 << 20)
    assert len(dps) > 4000
    items = []
    for x, dd, k, _j in dps:
        biased = (dd + wdiv2) % kgo.N if k & 1 else dd
        items.append(struct.pack("<QQQQQQQ", *[(x >> (64 * i)) & M64 for i in range(4)], biased & M64, (biased >> 64) & M64, k))
    t = DPTable(threads=4)
    t.add_items(b"".join(items), wdiv2)
    n = len(t)
    assert n > 4000
    path = str(tmp_path / "kgx.work")
    t.save_work(path, 6, start, end, pub, total_count=2048 * 256, total_time=1.5)
    golden = json.load(open(os.path.join(ROOT, "tests", "golden", "work_file_golden.json")))
    data = open(path, "rb").read()
    assert (n, len(data)) == (golden["dp_count"], golden["bytes"])
    assert hashlib.sha256(data).hexdigest() == golden["sha256"]
    if os.path.exists(REFBIN):
        out = subprocess.run([REFBIN, "-winfo", path], capture_output=True, text=True, timeout=120).stdout
        assert str(n) in out and "DP" in out, out
        out = subprocess.run([REFBIN, "-wcheck", path], capture_output=True, text=True, timeout=300).stdout
        assert "[100.000% OK]" in out and "Wrong" not in out, out[-1500:]  # Check.cpp:393-409
    # and the file loads back into an identical table
    t2 = DPTable(threads=2, max_events=1 << 16)
    assert t2.load_work(path)[0] == 6 and len(t2) == n
    assert len(t2.add_items(b"".join(items), wdiv2)) == len(items)         # all duplicates now
    t.close(); t2.close()


def test_insert_rate_is_reported(oracle, capsys):
    from kangaroo_b200.ingest import DPTable
    rng = np.random.default_rng(3)
    n = 400000
    raw = np.zeros((n, 10), dtype=np.uint32)
    raw[:, 0] = np.arange(n)
    raw[:, 2:10] = rng.integers(0, 1 << 32, size=(n, 8), dtype=np.uint32)
    raw[:, 1] = raw[:, 6] & 0x3FFFF          # any bucket assignment is valid for the table; real records use x.bits64[2]
    raw[:, 9] &= 0x3FFFFFFF
    for threads in (1, 4):
        t = DPTable(threads=threads)
        t0 = time.perf_counter()
        for c in range(0, n, 50000):
            t.add_dp40(raw[c:c + 50000])
        dt = time.perf_counter() - t0
        assert len(t) == n
        with capsys.disabled():
            print("\n[ingest] %d threads: %.2f M DP/s (%d records, batches of 50000)" % (threads, n / dt / 1e6, n))
        t.close()


def test_small_search_end_to_end_on_the_cpu(oracle):
    """The whole host side of a search without a GPU: herds and jumps from the oracle (SolveKeyCPU's loop, Kangaroo.cpp:375-433),
    every distinguished point through kgi_add into the reference's HashTable, same-herd hits answered by re-creating that
    kangaroo (Kangaroo.cpp:601-609), the tame/wild collision resolved by the reference's CheckKey -> the private key."""
    from kangaroo_b200.ingest import DPTable, EV_RESET, EV_COLLISION
    rp, dp_bits, n = 32, 5, 256
    start = 0x49DCCFD96DC5DF56487436F5A1B18C4F5D34F65DDB48CB5E0000000000000000
    oracle.rseed(0x600DCAFE)
    priv = start + oracle.rand_bits(rp)
    key = ec.add(ec.mul(priv), ec.neg(ec.mul(start)))
    table = oracle.create_jump_table(rp)
    wd2 = 1 << (rp - 1)
    px, py, d = oracle.create_herd(n, rp, wd2, key)
    mask = oracle.dp_mask(dp_bits)
    t = DPTable(threads=2, max_events=1 << 14)
    found, jumps, resets = None, 0, 0
    for _ in range(400):                                                  # 400 x 256 x 64 = 6.5 M jumps >> 2 sqrt(2^32)
        dps = oracle.jump_cpu(px, py, d, table, 64, mask)
        jumps += n * 64
        ev = t.add_dp40(b"".join(rec40(oracle, x, dist, kidx & 1, kidx) for x, dist, kidx, _ in dps))
        for kind, _, kidx, d_old, d_new in ev:
            if kind == EV_COLLISION:
                found = t.resolve(d_old, d_new, key, start)
            elif kind == EV_RESET:
                resets += 1
                nx, ny, nd = oracle.create_herd(1, rp, wd2, key, first_type=kidx & 1)
                px[kidx], py[kidx], d[kidx] = nx[0], ny[0], nd[0]
        if found is not None:
            break
    t.close()
    print("solved after %d jumps (2 sqrt(N) = %d), %d resets" % (jumps, 2 << (rp // 2), resets))
    assert found == priv
