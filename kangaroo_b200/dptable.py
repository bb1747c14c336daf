"""Rank-0 distinguished-point table in device memory (C ABI: include/kgx.h kgx_dpt_*, kernels in csrc/kgx_dptable.cuh), and
the rule that picks it or the host table (ingest.DPTable) for a run.

The device table makes the decisions of the host table's kgi_add (the reference's HashTable::Add) on the DP records where
they already are -- the gather buffer on rank 0 -- so a run at a low dp is not held back by a CPU inserting 600 k records per
step.  Its content reaches a work file through an export in work-file order and kgi_fill_sorted; a resumed file reaches it
through kgi_export_sorted and a bulk load.  No Python-side fallback: without libkgx.so DeviceDPTable() raises."""
import ctypes
import math
import os

import numpy as np

from ._lib import load_library
from .ingest import Event

HASH_SIZE = 1 << 18
Z0 = 2.0 * (2.0 - math.sqrt(2.0)) * math.sqrt(math.pi)
CAP_FLOOR = 1 << 20            # smallest device table the solver allocates
EXPORT_CHUNK = 1 << 22         # entries per export / load chunk (the library's scratch)
_u64p = ctypes.POINTER(ctypes.c_uint64)


def compute_expected(range_power, kangaroos, dp):
    """Kangaroo::ComputeExpected (Kangaroo.cpp:836-873, without symmetry): expected jumps to a solve with `kangaroos` walks
    in total at `dp` bits, and its ratio to the dp-0 expectation Z0*sqrt(N)."""
    n = 2.0 ** range_power
    ops = Z0 * (n * (kangaroos * 2.0 ** dp + math.sqrt(n))) ** (1.0 / 3.0)
    return ops, ops / (Z0 * math.sqrt(n))


def suggested_dp(range_power, kangaroos):
    """The reference's "Suggested DP" (Kangaroo.cpp:984-991): the largest dp whose overhead is at most 5 %."""
    dp = max(int(range_power / 2.0 - math.log2(kangaroos)), 0)
    while dp > 0 and compute_expected(range_power, kangaroos, dp)[1] > 1.05:
        dp -= 1
    return dp


def memory_bytes(capacity):
    """device bytes a table of `capacity` entries holds (kgx_dpt_memory_bytes)"""
    return int(load_library().kgx_dpt_memory_bytes(int(capacity)))


def max_capacity():
    return int(load_library().kgx_dpt_max_capacity())


def budget_capacity(free_bytes):
    """largest capacity whose table, export scratch included, fits in 3/4 of `free_bytes` (0 when none does)"""
    budget = 0.75 * free_bytes
    lo, hi = 0, max_capacity()
    if memory_bytes(1) > budget:
        return 0
    while lo < hi:
        mid = (lo + hi + 1) // 2
        if memory_bytes(mid) <= budget:
            lo = mid
        else:
            hi = mid - 1
    return lo


def choose_table(expected_entries, free_bytes, mode="auto", cap=None):
    """The table a run uses -> ("device", capacity) or ("host", 0).
    auto: capacity = min(budget, 2 E) (at least CAP_FLOOR), the device table when that holds at least 1.5 E entries and fits
    the budget (3/4 of the free device memory); mode "host" / "device" pins the kind, `cap` pins the capacity."""
    if mode not in ("auto", "host", "device"):
        raise ValueError("KGX_DPTABLE must be auto, host or device, not %r" % mode)
    if mode == "host":
        return "host", 0
    budget = budget_capacity(free_bytes)
    if cap is None:
        cap = min(max(min(budget, int(2 * expected_entries)), CAP_FLOOR), max_capacity())
    if mode == "device" or (cap >= 1.5 * expected_entries and cap <= budget):
        return "device", int(cap)
    return "host", 0


def choose_from_env(expected_entries, free_bytes):
    """choose_table with KGX_DPTABLE=auto|host|device and KGX_DPTABLE_CAP=<entries> from the environment"""
    cap = os.environ.get("KGX_DPTABLE_CAP")
    return choose_table(expected_entries, free_bytes, os.environ.get("KGX_DPTABLE", "auto") or "auto",
                        int(cap) if cap else None)


class DeviceDPTable:
    """kgx_dpt_*: inserts stream-ordered on the caller's stream, events one insert later, exports in work-file order."""

    def __init__(self, dev, capacity, max_events=4096):
        self._lib = load_library()
        h = self._lib.kgx_dpt_create(int(dev), int(capacity), int(max_events))
        if not h:
            raise RuntimeError("DeviceDPTable: %s" % self._lib.kgx_dpt_last_error(None).decode())
        self._h = ctypes.c_void_p(h)
        self.capacity = int(capacity)
        self._ev = (Event * max_events)()
        self._cap = max_events
        self.entries = 0                 # after the last insert whose events were collected
        self._inflight = []              # records of the inserts whose events were not collected yet
        self._exp = None                 # host buffers of an export

    def _ck(self, rc, what):
        if rc != 0:
            raise RuntimeError("DeviceDPTable.%s: %s" % (what, self._lib.kgx_dpt_last_error(self._h).decode()))

    def close(self):
        if self._h:
            self._lib.kgx_dpt_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def memory(self):
        return memory_bytes(self.capacity)

    @property
    def pending(self):
        return len(self._inflight)

    def fits(self, n):
        """True when n more records cannot take the table past its capacity, whatever the pending inserts add"""
        return self.entries + sum(self._inflight) + n <= self.capacity

    def insert(self, ptr, counts, stride=0, stream=0):
        """Queue the records of one step: rank r's counts[r] 40-byte records at device address ptr + r * stride * 40, on
        `stream` (a cudaStream_t as int; 0 = the legacy default stream).  At most two inserts may await events()."""
        c = (ctypes.c_uint32 * len(counts))(*[int(v) for v in counts])
        self._ck(self._lib.kgx_dpt_insert(self._h, ctypes.c_void_p(int(ptr)), int(stride), c, len(counts), ctypes.c_void_p(int(stream))),
                 "insert")
        self._inflight.append(sum(int(v) for v in counts))

    def events(self):
        """events of the oldest pending insert (waits for it) -> list of (kind, rank, kidx, d_old, d_new), as DPTable.add_dp40"""
        ne, ent = ctypes.c_uint32(0), ctypes.c_uint64(0)
        rc = self._lib.kgx_dpt_events(self._h, ctypes.cast(self._ev, ctypes.c_void_p), self._cap, ctypes.byref(ne), ctypes.byref(ent))
        if rc == -3:
            self._ck(rc, "events")
        self._inflight.pop(0)
        self.entries = int(ent.value)
        if rc == -1:
            raise RuntimeError("kgx_dpt_insert: malformed DP record (h >= 2^18)")
        if rc == -2:
            raise RuntimeError("kgx_dpt_insert: %s" % self._lib.kgx_dpt_last_error(self._h).decode())
        out = []
        for i in range(min(ne.value, self._cap)):
            e = self._ev[i]
            out.append((int(e.kind), int(e.rank), int(e.kidx), (int(e.d_old[0]), int(e.d_old[1])), (int(e.d_new[0]), int(e.d_new[1]))))
        return out

    def count(self):
        """entries after every queued insert (waits for them)"""
        v = ctypes.c_uint64(0)
        self._ck(self._lib.kgx_dpt_count(self._h, ctypes.byref(v)), "count")
        return int(v.value)

    def __len__(self):
        return self.count()

    # -- export: a snapshot of the inserts queued before export_begin, read in chunks from any thread ----------------------
    def export_begin(self, stream=0):
        self._ck(self._lib.kgx_dpt_export_begin(self._h, ctypes.c_void_p(int(stream))), "export_begin")

    def export_chunks(self, chunk=EXPORT_CHUNK):
        """yields (h uint32 [k], entries uint64 [k, 4]) in work-file order; the arrays are reused between chunks"""
        if self._exp is None or self._exp[0].shape[0] != chunk:
            self._exp = (np.empty((chunk, 4), dtype=np.uint64), np.empty(4096, dtype=np.uint32))
        ent, counts = self._exp
        first = 0
        nb, ne = ctypes.c_uint32(0), ctypes.c_uint64(0)
        while first < HASH_SIZE:
            self._ck(self._lib.kgx_dpt_export_read(self._h, first, HASH_SIZE - first, ctypes.c_void_p(ent.ctypes.data), chunk,
                                                   ctypes.c_void_p(counts.ctypes.data), ctypes.byref(nb), ctypes.byref(ne)),
                     "export_read")
            k, n = nb.value, ne.value
            if n:
                yield np.repeat(np.arange(first, first + k, dtype=np.uint32), counts[:k]), ent[:n]
            first += k

    def export_end(self):
        self._ck(self._lib.kgx_dpt_export_end(self._h), "export_end")

    def export_to_host(self, host):
        """Fill the host table `host` (ingest.DPTable, reset first) with the export begun last; ends the export."""
        try:
            host.reset()
            for h, e in self.export_chunks():
                host.fill_sorted(h, e)
        finally:
            self.export_end()

    def to_host(self, host, stream=0):
        """the whole table as it is after the inserts queued so far -> host table"""
        self.export_begin(stream)
        self.export_to_host(host)

    # -- bulk load (resume) ---------------------------------------------------------------------------------------------
    def load(self, h, entries):
        h = np.ascontiguousarray(h, dtype=np.uint32)
        e = np.ascontiguousarray(entries, dtype=np.uint64).reshape(-1, 4)
        assert h.shape[0] == e.shape[0]
        if self.entries + h.shape[0] > self.capacity:
            raise RuntimeError("DeviceDPTable.load: %d entries do not fit a table of %d" % (self.entries + h.shape[0], self.capacity))
        self._ck(self._lib.kgx_dpt_load(self._h, ctypes.c_void_p(h.ctypes.data), ctypes.c_void_p(e.ctypes.data), h.shape[0]), "load")
        self.entries += h.shape[0]

    def load_from_host(self, host, chunk=EXPORT_CHUNK):
        """every entry of the host table (kgi_export_sorted) -> this table"""
        n, first = len(host), 0
        while first < n:
            h, e = host.export_sorted(first, min(chunk, n - first))
            self.load(h, e)
            first += h.shape[0]
