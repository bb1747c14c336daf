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

    def load_work(self, path):
        dp, cnt, tm = ctypes.c_uint32(0), ctypes.c_uint64(0), ctypes.c_double(0)
        rc = self._lib.kgi_load_work(self._h, os.fsencode(path), ctypes.byref(dp), ctypes.byref(cnt), ctypes.byref(tm))
        if rc != 0:
            raise RuntimeError("kgi_load_work: %s is not a HEADW work file" % path)
        return dp.value, cnt.value, tm.value
