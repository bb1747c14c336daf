"""ctypes binding of csrc/libkgx_ingest.so (C ABI: include/kgx_ingest.h): the rank-0 distinguished-point table.

The table follows the reference's `class HashTable` (HashTable.{h,cpp}: same insert semantics, same work-file layout) and
is filled by a batched, bucket-sharded multi-threaded insert that replaces the single-mutex loop of Kangaroo::SolveKeyGPU
(Kangaroo.cpp:594-612) when the DP records of all GPUs arrive on rank 0.
No Python-side fallback: without the library DPTable() raises."""
import ctypes
import os

import numpy as np

from ._lib import INGEST_PATH as LIB_PATH

EV_RESET, EV_COLLISION = 1, 2
DP40_BYTES, ITEM_BYTES = 40, 56
WALK_BYTES = 96          # work-file kangaroo record {x[4], y[4], d[4]}
_M64 = 0xFFFFFFFFFFFFFFFF


class Event(ctypes.Structure):
    """kgi_event"""
    _fields_ = [("kind", ctypes.c_uint32), ("rank", ctypes.c_uint32), ("kidx", ctypes.c_uint32), ("h", ctypes.c_uint32),
                ("d_old", ctypes.c_uint64 * 2), ("d_new", ctypes.c_uint64 * 2)]


_u64p = ctypes.POINTER(ctypes.c_uint64)
_SIGS = {
    "kgi_create": (ctypes.c_void_p, [ctypes.c_int]),
    "kgi_destroy": (None, [ctypes.c_void_p]),
    "kgi_reset": (None, [ctypes.c_void_p]),
    "kgi_count": (ctypes.c_uint64, [ctypes.c_void_p]),
    "kgi_threads": (ctypes.c_int, [ctypes.c_void_p]),
    "kgi_add": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint32, ctypes.c_uint32, ctypes.POINTER(Event), ctypes.c_uint32,
                               ctypes.POINTER(ctypes.c_uint32)]),
    "kgi_add_items": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint32, ctypes.c_uint32, _u64p, ctypes.POINTER(Event),
                                     ctypes.c_uint32, ctypes.POINTER(ctypes.c_uint32)]),
    "kgi_resolve": (ctypes.c_int, [ctypes.c_void_p, _u64p, _u64p, _u64p, _u64p, _u64p, _u64p]),
    "kgi_save_work": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_char_p, ctypes.c_uint32, _u64p, _u64p, _u64p, _u64p, ctypes.c_uint64,
                                     ctypes.c_double]),
    "kgi_load_work": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_char_p, ctypes.POINTER(ctypes.c_uint32), _u64p,
                                     ctypes.POINTER(ctypes.c_double)]),
    "kgi_save_work_walks": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_char_p, ctypes.c_uint32, _u64p, _u64p, _u64p, _u64p,
                                           ctypes.c_uint64, ctypes.c_double, ctypes.c_uint64, _u64p]),
    "kgi_load_work_ex": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_char_p, ctypes.POINTER(ctypes.c_uint32), _u64p, _u64p, _u64p, _u64p,
                                        _u64p, ctypes.POINTER(ctypes.c_double), _u64p, _u64p]),
    "kgi_fill_sorted": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint64]),
    "kgi_export_sorted": (ctypes.c_uint64, [ctypes.c_void_p, ctypes.c_uint64, ctypes.c_uint64, ctypes.c_void_p, ctypes.c_void_p]),
}
EXPORTED_SYMBOLS = sorted(_SIGS)
_lib = None


def load_library():
    global _lib
    if _lib is not None:
        return _lib
    path = os.path.abspath(LIB_PATH)
    if not os.path.exists(path):
        raise RuntimeError("kangaroo_b200: %s is missing (run __graft_entry__.build())" % path)
    lib = ctypes.CDLL(path)
    for name, (res, args) in _SIGS.items():
        fn = getattr(lib, name)
        fn.restype, fn.argtypes = res, args
    _lib = lib
    return lib


def _limbs4(v):
    return (ctypes.c_uint64 * 4)(*[(int(v) >> (64 * k)) & _M64 for k in range(4)])


def _int4(a):
    return sum(int(a[k]) << (64 * k) for k in range(4))


class WorkInfo:
    """Header of a HEADW work file (Backup.cpp:154-200) plus where its kangaroos are."""
    __slots__ = ("path", "dp_bits", "range_start", "range_end", "key", "total_count", "total_time", "n_walks", "walk_offset")

    def __init__(self, **kw):
        for k, v in kw.items():
            setattr(self, k, v)

    def __repr__(self):
        return "WorkInfo(%s)" % ", ".join("%s=%r" % (k, getattr(self, k)) for k in self.__slots__)


def read_work_info(path, table=None):
    """Read a work file's header and walk count (kgi_load_work_ex); load its DP table into `table` (a DPTable) when
    given, else skip the table.  Raises ValueError when the key is not on the curve."""
    lib = load_library()
    dp, cnt, tm = ctypes.c_uint32(0), ctypes.c_uint64(0), ctypes.c_double(0)
    rs, re, kx, ky = ((ctypes.c_uint64 * 4)() for _ in range(4))
    nw, off = ctypes.c_uint64(0), ctypes.c_uint64(0)
    rc = lib.kgi_load_work_ex(table._h if table is not None else None, os.fsencode(path), ctypes.byref(dp), rs, re, kx, ky,
                              ctypes.byref(cnt), ctypes.byref(tm), ctypes.byref(nw), ctypes.byref(off))
    if rc == -2:
        raise ValueError("%s: key does not lie on the elliptic curve" % path)
    if rc != 0:
        raise RuntimeError("kgi_load_work_ex: %s is not a HEADW work file" % path)
    return WorkInfo(path=path, dp_bits=dp.value, range_start=_int4(rs), range_end=_int4(re), key=(_int4(kx), _int4(ky)),
                    total_count=cnt.value, total_time=tm.value, n_walks=nw.value, walk_offset=off.value)


class DPTable:
    """Rank-0 DP table: HashTable semantics + sharded batched insert (Kangaroo::AddToTable semantics per record)."""

    def __init__(self, threads=0, max_events=4096):
        self._lib = load_library()
        self._h = ctypes.c_void_p(self._lib.kgi_create(int(threads)))
        if not self._h:
            raise RuntimeError("kgi_create failed")
        self._ev = (Event * max_events)()
        self._cap = max_events
        self.threads = self._lib.kgi_threads(self._h)

    def close(self):
        if self._h:
            self._lib.kgi_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __len__(self):
        return int(self._lib.kgi_count(self._h))

    def reset(self):
        self._lib.kgi_reset(self._h)

    def _events(self, n):
        out = []
        for i in range(min(n, self._cap)):
            e = self._ev[i]
            out.append((int(e.kind), int(e.rank), int(e.kidx), (int(e.d_old[0]), int(e.d_old[1])), (int(e.d_new[0]), int(e.d_new[1]))))
        return out

    @staticmethod
    def _buf(buf, rec):
        a = np.ascontiguousarray(np.frombuffer(buf, dtype=np.uint8) if not isinstance(buf, np.ndarray) else buf.view(np.uint8).reshape(-1))
        assert a.size % rec == 0
        return a, a.size // rec

    def add_dp40(self, buf, rank=0):
        """buf: n x 40-byte DP records (bytes / uint8 ndarray) -> list of (kind, rank, kidx, d_old, d_new) events."""
        a, n = self._buf(buf, DP40_BYTES)
        ne = ctypes.c_uint32(0)
        rc = self._lib.kgi_add(self._h, a.ctypes.data_as(ctypes.c_void_p), n, int(rank), self._ev, self._cap, ctypes.byref(ne))
        if rc != 0:
            raise RuntimeError("kgi_add: malformed DP record (h >= 2^18)")
        return self._events(ne.value)

    def add_items(self, buf, wild_offset, rank=0):
        """buf: n x 56-byte engine ITEMs (biased distances) -> events; HashTable::Convert applied on the host."""
        a, n = self._buf(buf, ITEM_BYTES)
        wo = (ctypes.c_uint64 * 2)(int(wild_offset) & _M64, (int(wild_offset) >> 64) & _M64)
        ne = ctypes.c_uint32(0)
        rc = self._lib.kgi_add_items(self._h, a.ctypes.data_as(ctypes.c_void_p), n, int(rank), wo, self._ev, self._cap, ctypes.byref(ne))
        if rc != 0:
            raise RuntimeError("kgi_add_items failed")
        return self._events(ne.value)

    def resolve(self, d_old, d_new, key, range_start):
        """Kangaroo::CollisionCheck/CheckKey -> private key (int) or None."""
        a = (ctypes.c_uint64 * 2)(*d_old); b = (ctypes.c_uint64 * 2)(*d_new)
        out = (ctypes.c_uint64 * 4)()
        rc = self._lib.kgi_resolve(self._h, a, b, _limbs4(key[0]), _limbs4(key[1]), _limbs4(range_start), out)
        return sum(int(out[k]) << (64 * k) for k in range(4)) if rc == 1 else None

    def save_work(self, path, dp_bits, range_start, range_end, pubkey, total_count=0, total_time=0.0):
        rc = self._lib.kgi_save_work(self._h, os.fsencode(path), int(dp_bits), _limbs4(range_start), _limbs4(range_end),
                                     _limbs4(pubkey[0]), _limbs4(pubkey[1]), int(total_count), float(total_time))
        if rc != 0:
            raise RuntimeError("kgi_save_work: cannot write %s" % path)

    def save_work_walks(self, path, dp_bits, range_start, range_end, pubkey, total_count, total_time, total_walks):
        """save_work with `total_walks` kangaroo records to follow; the file already has its final size.  Returns the byte
        offset of the first walk record."""
        off = ctypes.c_uint64(0)
        rc = self._lib.kgi_save_work_walks(self._h, os.fsencode(path), int(dp_bits), _limbs4(range_start), _limbs4(range_end),
                                           _limbs4(pubkey[0]), _limbs4(pubkey[1]), int(total_count), float(total_time),
                                           int(total_walks), ctypes.byref(off))
        if rc != 0:
            raise RuntimeError("kgi_save_work_walks: cannot write %s" % path)
        return off.value

    def load_work_ex(self, path):
        """load_work returning the whole header (WorkInfo)."""
        return read_work_info(path, self)

    def fill_sorted(self, h, entries):
        """Append entries given in work-file order (kgi_fill_sorted): h uint32 [n], entries uint64 [n, 4] = {x[2], d[2]}."""
        h = np.ascontiguousarray(h, dtype=np.uint32)
        e = np.ascontiguousarray(entries, dtype=np.uint64).reshape(-1, 4)
        assert h.shape[0] == e.shape[0]
        if self._lib.kgi_fill_sorted(self._h, h.ctypes.data_as(ctypes.c_void_p), e.ctypes.data_as(ctypes.c_void_p), h.shape[0]) != 0:
            raise RuntimeError("kgi_fill_sorted: entries out of work-file order or h >= 2^18")

    def export_sorted(self, first=0, n=None):
        """Entries [first, first + n) in work-file order (kgi_export_sorted) -> (h uint32 [k], entries uint64 [k, 4])."""
        n = len(self) - first if n is None else n
        h = np.empty(max(n, 0), dtype=np.uint32)
        e = np.empty((max(n, 0), 4), dtype=np.uint64)
        k = int(self._lib.kgi_export_sorted(self._h, int(first), max(n, 0), h.ctypes.data_as(ctypes.c_void_p),
                                            e.ctypes.data_as(ctypes.c_void_p)))
        return h[:k], e[:k]

    def load_work(self, path):
        dp, cnt, tm = ctypes.c_uint32(0), ctypes.c_uint64(0), ctypes.c_double(0)
        rc = self._lib.kgi_load_work(self._h, os.fsencode(path), ctypes.byref(dp), ctypes.byref(cnt), ctypes.byref(tm))
        if rc != 0:
            raise RuntimeError("kgi_load_work: %s is not a HEADW work file" % path)
        return dp.value, cnt.value, tm.value
