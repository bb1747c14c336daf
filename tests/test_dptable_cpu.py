"""CPU checks of the pieces around the device DP table: the host table's bulk paths in work-file order (kgi_fill_sorted,
kgi_export_sorted), the port of Kangaroo::ComputeExpected / "Suggested DP", and the rule that picks the table kind."""
import math

import numpy as np
import pytest

from kangaroo_b200 import dptable
from kangaroo_b200.ingest import DPTable

DP40 = np.dtype([("kidx", "<u4"), ("h", "<u4"), ("x", "<u8", 2), ("d", "<u8", 2)])
KEY = (0x79BE667EF9DCBBAC55A06295CE870B07029BFCDB2DCE28D959F2815B16F81798,
       0x483ADA7726A3C4655DA4FBFC0E1108A8FD17B448A68554199C47D08FFB10D4B8)


def stream(n, seed, buckets=64):
    """n records with distinct x (duplicate-free), crowded into a few buckets so that caps grow past 16"""
    rng = np.random.default_rng(seed)
    r = np.zeros(n, dtype=DP40)
    r["kidx"] = rng.integers(0, 1 << 20, n)
    r["h"] = rng.integers(0, buckets, n)
    r["x"] = rng.integers(0, 1 << 63, (n, 2), dtype=np.uint64) * np.uint64(2) + np.uint64(1)
    r["d"] = rng.integers(0, 1 << 63, (n, 2), dtype=np.uint64)
    return r


def sorted_entries(recs):
    o = np.lexsort((recs["x"][:, 0], recs["x"][:, 1], recs["h"]))
    s = recs[o]
    return s["h"].copy(), np.concatenate([s["x"], s["d"]], axis=1).astype(np.uint64)


def save(table, path):
    table.save_work(str(path), 12, 1 << 40, (1 << 41) - 1, KEY, total_count=123, total_time=4.5)
    return open(path, "rb").read()


@pytest.mark.parametrize("chunks", [1, 7])
def test_fill_sorted_matches_sequential_adds(tmp_path, chunks):
    recs = stream(6000, 1)
    a = DPTable(threads=4)
    for part in np.array_split(recs, 5):                       # several batches, like steps
        assert a.add_dp40(part.view(np.uint8)) == []
    want = save(a, tmp_path / "a.work")
    h, e = sorted_entries(recs)
    b = DPTable(threads=1)
    b.reset()
    for ph, pe in zip(np.array_split(h, chunks), np.array_split(e, chunks)):
        b.fill_sorted(ph, pe)
    assert len(b) == len(recs)
    assert save(b, tmp_path / "b.work") == want
    a.close(); b.close()


def test_fill_sorted_refuses_bad_order():
    recs = stream(100, 2, buckets=4)
    h, e = sorted_entries(recs)
    t = DPTable(threads=1)
    with pytest.raises(RuntimeError):
        t.fill_sorted(h[::-1], e[::-1])
    assert len(t) == 0                                         # a refused chunk changes nothing
    t.fill_sorted(h[:50], e[:50])
    with pytest.raises(RuntimeError):
        t.fill_sorted(h[:1], e[:1])                            # x not above what the bucket already holds
    bad = h.copy(); bad[-1] = 1 << 18
    with pytest.raises(RuntimeError):
        t.fill_sorted(bad[50:], e[50:])
    t.fill_sorted(h[50:], e[50:])
    assert len(t) == 100
    t.close()


def test_export_sorted_round_trip(tmp_path):
    recs = stream(5000, 3, buckets=1 << 18)
    a = DPTable(threads=2)
    a.add_dp40(recs.view(np.uint8))
    h, e = a.export_sorted()
    wh, we = sorted_entries(recs)
    assert np.array_equal(h, wh) and np.array_equal(e, we)
    parts = [a.export_sorted(f, 700) for f in range(0, 5000, 700)]
    assert np.array_equal(np.concatenate([p[0] for p in parts]), wh)
    assert np.array_equal(np.concatenate([p[1] for p in parts]), we)
    assert a.export_sorted(5000, 10)[0].size == 0
    b = DPTable(threads=1)
    b.fill_sorted(h, e)
    assert save(b, tmp_path / "b.work") == save(a, tmp_path / "a.work")
    a.close(); b.close()


def _reference_expected(range_power, k, dp):
    """Kangaroo::ComputeExpected written out from the formula: Z0 (N (k 2^dp + sqrt N))^(1/3), Z0 = 2 (2 - sqrt 2) sqrt pi"""
    n = 2.0 ** range_power
    return 2 * (2 - math.sqrt(2)) * math.sqrt(math.pi) * (n * (k * 2 ** dp + math.sqrt(n))) ** (1 / 3)


@pytest.mark.parametrize("rp,k,dp", [(80, 8 * 4849664, 16), (80, 8 * 4849664, 12), (56, 32 * 128 * 128, 8), (110, 2 ** 20, 0)])
def test_compute_expected(rp, k, dp):
    ops, over = dptable.compute_expected(rp, k, dp)
    assert ops == pytest.approx(_reference_expected(rp, k, dp), rel=1e-12)
    assert over == pytest.approx(ops / (2.077 * 2 ** (rp / 2)), rel=1e-3)


def test_suggested_dp_flagship():
    k = 8 * 4849664                                            # 8 GPUs x the default grid
    assert dptable.suggested_dp(80, k) == 12
    assert math.log2(dptable.compute_expected(80, k, 16)[0]) == pytest.approx(41.63, abs=0.01)
    assert math.log2(dptable.compute_expected(80, k, 12)[0]) == pytest.approx(41.12, abs=0.01)
    assert dptable.suggested_dp(20, 2 ** 20) == 0


def test_choose_table():
    per = dptable.memory_bytes(1 << 30) / (1 << 30)
    assert 40 / 0.7 * 0.99 < per < 100                         # one slot and its load factor cost under 100 B per entry
    e = 10 ** 8
    free = 180e9
    kind, cap = dptable.choose_table(e, free)
    assert kind == "device" and cap == 2 * e
    # the budget (3/4 of free memory) holds 1.5 E but not 2 E: device, capacity = budget
    free = dptable.memory_bytes(int(1.7 * e)) / 0.75
    kind, cap = dptable.choose_table(e, free)
    assert kind == "device" and 1.5 * e <= cap < 2 * e and dptable.memory_bytes(cap) <= 0.75 * free
    free = dptable.memory_bytes(int(1.4 * e)) / 0.75           # under 1.5 E: host
    assert dptable.choose_table(e, free) == ("host", 0)
    assert dptable.choose_table(e, free, mode="device")[0] == "device"
    assert dptable.choose_table(e, 180e9, mode="host") == ("host", 0)
    assert dptable.choose_table(10, 180e9) == ("device", dptable.CAP_FLOOR)
    assert dptable.choose_table(10000, 180e9, cap=5000) == ("host", 0)   # a pinned capacity below 1.5 E
    assert dptable.choose_table(10000, 180e9, mode="device", cap=5000) == ("device", 5000)
    assert dptable.choose_table(1e12, 180e9) == ("host", 0)
    with pytest.raises(ValueError):
        dptable.choose_table(10, 1e9, mode="gpu")
