"""Host-side mirror of the reference's `class GPUEngine` (GPU/GPUEngine.h:40-84) over the C ABI.

Same method names, argument meaning and error behaviour as the reference class so the parity tests read like
Check.cpp:467-621.  Where the reference passes `Int*` arrays this mirror takes Python ints (or numpy uint64
limb arrays); the wild-offset bookkeeping that GPUEngine.cu does on the host with Int::ModAddK1order /
ModSubK1order (GPUEngine.cu:407-411, 477, 526, 672) is done here mod n.  All device work happens in libkgx.so.
"""
import ctypes

import numpy as np

from ._lib import Item, load_library

NB_JUMP = 32        # Constants.h:29
GPU_GRP_SIZE = 128  # Constants.h:32
NB_RUN = 64         # Constants.h:35
TAME, WILD = 0, 1   # Constants.h:38-39
WALK_SIZE = 96      # work-file kangaroo record {x[4], y[4], d[4]} (Backup.cpp:535-545)
ORDER = 0xFFFFFFFFFFFFFFFFFFFFFFFFFFFFFFFEBAAEDCE6AF48A03BBFD25E8CD0364141
_M64 = 0xFFFFFFFFFFFFFFFF
_u64p = ctypes.POINTER(ctypes.c_uint64)


class ITEM:
    """GPUEngine.h:34-38: {Int x; Int d; uint64_t kIdx}"""
    __slots__ = ("x", "d", "kIdx")

    def __init__(self, x, d, kIdx):
        self.x, self.d, self.kIdx = x, d, kIdx

    def __repr__(self):
        return "ITEM(x=%x, d=%x, kIdx=%d)" % (self.x, self.d, self.kIdx)


def _limbs(vals, limbs):
    """list of ints / (n,limbs) array -> contiguous (n,limbs) uint64"""
    if isinstance(vals, np.ndarray):
        a = np.ascontiguousarray(vals, dtype=np.uint64)
        assert a.ndim == 2 and a.shape[1] >= limbs
        return np.ascontiguousarray(a[:, :limbs])
    out = np.empty((len(vals), limbs), dtype=np.uint64)
    for i, v in enumerate(vals):
        for k in range(limbs):
            out[i, k] = (v >> (64 * k)) & _M64
    return out


def _ints(a):
    a = np.asarray(a, dtype=np.uint64)
    obj = a.astype(object)
    acc = obj[:, 0]
    for k in range(1, a.shape[1]):
        acc = acc + (obj[:, k] << (64 * k))
    return [int(v) for v in acc]


def _p(a):
    return a.ctypes.data_as(_u64p)


class GPUEngine:
    KERNELS = {"auto": 0, "stream": 1, "resident": 2, "tmem": 3}

    def __init__(self, nbThreadGroup, nbThreadPerGroup, gpuId=0, maxFound=65536, kernel="auto", stream_g=0):
        """kernel / stream_g are not in the reference constructor (GPUEngine.cu:144): they pin the jump kernel
        (kgx_create_ex) so that the parity tests can run every case on both; "auto" is the product default."""
        self._lib = load_library()
        self._h = None
        self.initialised = False
        self.wildOffset = 0
        self.nbThreadPerGroup = nbThreadPerGroup
        self.nbThread = nbThreadGroup * nbThreadPerGroup
        self.maxFound = maxFound
        self.lostWarning = False
        h = self._lib.kgx_create_ex(gpuId, nbThreadGroup, nbThreadPerGroup, maxFound, self.KERNELS[kernel], int(stream_g))
        if not h:
            # the reference prints and leaves initialised=false (GPUEngine.cu:152-170); a Python mirror raising is the
            # loud equivalent -- there is no CPU path to fall back to.
            raise RuntimeError("GPUEngine: %s" % self._lib.kgx_last_error(None).decode())
        self._h = ctypes.c_void_p(h)
        buf = ctypes.create_string_buffer(256)
        self._lib.kgx_device_info(gpuId, buf, 256)
        name, sms, _, _, _ = buf.value.decode().split("|")
        self.deviceName = "GPU #%d %s (%sx%d cores) Grid(%dx%d)" % (gpuId, name, sms, 128, nbThreadGroup, nbThreadPerGroup)
        self._items = (Item * maxFound)()
        self.kernel = {1: "stream", 2: "resident", 3: "tmem"}[self._lib.kgx_kernel_kind(self._h)]
        self.initialised = True

    # -- bookkeeping -------------------------------------------------------------------------------------
    def _ck(self, rc, what):
        if rc != 0:
            raise RuntimeError("GPUEngine: %s: %s" % (what, self._lib.kgx_last_error(self._h).decode()))

    def close(self):
        if self._h:
            self._lib.kgx_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def GetNbThread(self):
        return self.nbThread

    def GetGroupSize(self):
        return GPU_GRP_SIZE

    def GetMemory(self):
        return int(self._lib.kgx_memory_bytes(self._h))

    @property
    def nbKangaroo(self):
        return self.nbThread * GPU_GRP_SIZE

    @staticmethod
    def GetGridSize(gpuId, x, y):
        lib = load_library()
        cx, cy = ctypes.c_int(x), ctypes.c_int(y)
        if lib.kgx_grid_default(gpuId, ctypes.byref(cx), ctypes.byref(cy)) != 0:
            return None
        return cx.value, cy.value

    # -- reference interface -----------------------------------------------------------------------------
    def SetWildOffset(self, offset):
        """GPUEngine.cu:140-142. Must be called before SetKangaroos."""
        self.wildOffset = int(offset)

    def SetParams(self, dpMask, distance, px, py):
        """GPUEngine.cu:559-590: distance uses bits64[0..1], points bits64[0..3]; arrays of NB_JUMP."""
        jd, jx, jy = _limbs(distance, 2), _limbs(px, 4), _limbs(py, 4)
        assert jd.shape[0] == NB_JUMP and jx.shape[0] == NB_JUMP and jy.shape[0] == NB_JUMP
        self.dpMask = dpMask
        self._ck(self._lib.kgx_set_params(self._h, ctypes.c_uint64(dpMask), _p(jd), _p(jx), _p(jy)), "SetParams")

    SYM_RULES = {None: 0, False: 0, "lastjump": 1, "symclass": 2, True: 2}

    def SetSymmetry(self, rule="symclass"):
        """USE_SYMMETRY engine mode (reference: compile-time Constants.h:25): equivalence-class switch on the device plus one of
        the reference's two jump rules -- "symclass" (SolveKeyCPU, Kangaroo.cpp:381-384) or "lastjump" (GPUCompute.h:53-58 =
        Check.cpp:536-541).  Distances cross the ABI as signed 128-bit values, the wild offset is not applied.  Before SetKangaroos."""
        mode = self.SYM_RULES[rule]
        self._ck(self._lib.kgx_set_symmetry(self._h, mode), "SetSymmetry")
        self.symmetry = mode != 0

    def _bias(self, d, kidx0=0):
        """+wildOffset mod n on odd kIdx (GPUEngine.cu:407-411), then truncate to 128 bits like the reference.
        Symmetric mode: d mod n -> signed 128-bit two's complement (values above n/2 are negative), no offset."""
        if getattr(self, "symmetry", False):
            return [((v - ORDER) if v > ORDER // 2 else v) & ((1 << 128) - 1) for v in d]
        out = []
        for i, v in enumerate(d):
            if (kidx0 + i) % 2 == WILD:
                v = (v + self.wildOffset) % ORDER
            out.append(v & ((1 << 128) - 1))
        return out

    def _unbias(self, v, kidx):
        if getattr(self, "symmetry", False):                          # signed 128-bit -> mod n
            return (v - (1 << 128)) % ORDER if v >> 127 else v
        return (v - self.wildOffset) % ORDER if kidx % 2 == WILD else v

    def SetKangaroos(self, px, py, d):
        """GPUEngine.cu:381-433; arrays of GetNbThread()*GPU_GRP_SIZE in kIdx order; d are ints mod n."""
        n = self.nbKangaroo
        ax, ay = _limbs(px, 4), _limbs(py, 4)
        dl = _ints(d) if isinstance(d, np.ndarray) else list(d)
        ad = _limbs(self._bias(dl), 2)
        assert ax.shape[0] == n and ay.shape[0] == n and ad.shape[0] == n
        self._ck(self._lib.kgx_upload(self._h, _p(ax), _p(ay), _p(ad)), "SetKangaroos")

    def GetKangaroos(self):
        """GPUEngine.cu:435-491 -> (px, py, d) lists of ints (d unbiased, mod n)."""
        n = self.nbKangaroo
        ax = np.empty((n, 4), dtype=np.uint64); ay = np.empty((n, 4), dtype=np.uint64); ad = np.empty((n, 2), dtype=np.uint64)
        self._ck(self._lib.kgx_download(self._h, _p(ax), _p(ay), _p(ad)), "GetKangaroos")
        d = [self._unbias(v, i) for i, v in enumerate(_ints(ad))]
        return _ints(ax), _ints(ay), d

    def GetKangaroosRaw(self):
        """numpy limb arrays, distances still biased (device convention)."""
        n = self.nbKangaroo
        ax = np.empty((n, 4), dtype=np.uint64); ay = np.empty((n, 4), dtype=np.uint64); ad = np.empty((n, 2), dtype=np.uint64)
        self._ck(self._lib.kgx_download(self._h, _p(ax), _p(ay), _p(ad)), "GetKangaroos")
        return ax, ay, ad

    def SnapshotBegin(self):
        """Asynchronous GetKangaroos (checkpoint path): snapshot after the launch in flight, do not block."""
        self._ck(self._lib.kgx_snapshot_begin(self._h), "SnapshotBegin")

    def SnapshotRead(self):
        """-> (px, py, d) lists of ints (d unbiased, mod n) of the snapshot taken by SnapshotBegin."""
        n = self.nbKangaroo
        ax = np.empty((n, 4), dtype=np.uint64); ay = np.empty((n, 4), dtype=np.uint64); ad = np.empty((n, 2), dtype=np.uint64)
        self._ck(self._lib.kgx_snapshot_read(self._h, _p(ax), _p(ay), _p(ad)), "SnapshotRead")
        return _ints(ax), _ints(ay), [self._unbias(v, i) for i, v in enumerate(_ints(ad))]

    def SetKangaroosRaw(self, ax, ay, ad):
        n = self.nbKangaroo
        ax, ay, ad = _limbs(ax, 4), _limbs(ay, 4), _limbs(ad, 2)
        assert ax.shape[0] == n
        self._ck(self._lib.kgx_upload(self._h, _p(ax), _p(ay), _p(ad)), "SetKangaroos")

    def SetKangaroo(self, kIdx, px, py, d):
        """GPUEngine.cu:493-538: patch one kangaroo (stream-ordered after any launch in flight)."""
        ax, ay = _limbs([px], 4), _limbs([py], 4)
        ad = _limbs(self._bias([d], kIdx), 2)
        self._ck(self._lib.kgx_patch(self._h, ctypes.c_uint64(kIdx), _p(ax), _p(ay), _p(ad)), "SetKangaroo")

    def CreateHerd(self, d, key):
        """Kangaroo::CreateHerd (Kangaroo.cpp:670-738) with the point arithmetic on the device: kangaroo i starts at
        d[i]*G (tame, even kIdx) or key + d[i]*G (wild, odd kIdx) -- the reference always builds the GPU herd with
        firstType = TAME (Kangaroo.cpp:540-545); d are ints mod n (wild ones already shifted by -rangeWidth/2 as the
        reference does).  Distances are stored biased like SetKangaroos."""
        firstType = TAME
        n = self.nbKangaroo
        dl = _ints(d) if isinstance(d, np.ndarray) else list(d)
        assert len(dl) == n
        sc = _limbs(dl, 4)
        ad = _limbs(self._bias(dl, firstType), 2)
        kx, ky = _limbs([key[0]], 4), _limbs([key[1]], 4)
        self._ck(self._lib.kgx_create_herd(self._h, _p(sc), _p(ad), _p(kx), _p(ky), int(firstType)), "CreateHerd")

    def CreateHerdRaw(self, scalars, d128, key):
        """CreateHerd from limb arrays: scalars (n,4) uint64 = d mod n (what the points are computed from),
        d128 (n,2) uint64 = the biased distances to store."""
        n = self.nbKangaroo
        sc, ad = _limbs(scalars, 4), _limbs(d128, 2)
        assert sc.shape[0] == n and ad.shape[0] == n
        kx, ky = _limbs([key[0]], 4), _limbs([key[1]], 4)
        self._ck(self._lib.kgx_create_herd(self._h, _p(sc), _p(ad), _p(kx), _p(ky), TAME), "CreateHerd")

    # -- work-file walks (kgx_walks_*: 96-byte {x[4], y[4], d[4]} records, d unbiased mod n) ----------------------
    def _wo(self):
        return _limbs([self.wildOffset & ((1 << 128) - 1)], 2)

    def WalksBegin(self):
        """Convert the herd into work-file records on the device, after the launch in flight; returns at once."""
        self._ck(self._lib.kgx_walks_begin(self._h, _p(self._wo())), "WalksBegin")

    def WalksRead(self, out, first=0, count=None):
        """Copy records [first, first + count) of the pending export into `out` (writable buffer of count * 96 bytes:
        numpy uint8 array or pinned torch tensor).  Waits for the export only."""
        count = self.nbKangaroo - first if count is None else count
        a = out if isinstance(out, np.ndarray) else None
        ptr = a.ctypes.data if a is not None else out.data_ptr()
        nbytes = a.nbytes if a is not None else out.numel() * out.element_size()
        assert nbytes >= count * WALK_SIZE
        self._ck(self._lib.kgx_walks_read(self._h, ctypes.c_void_p(ptr), int(first), int(count)), "WalksRead")
        return out

    def WalksEnd(self):
        self._ck(self._lib.kgx_walks_end(self._h), "WalksEnd")

    def GetWalks(self):
        """The whole herd as an (n, 12) uint64 array of work-file records (begin + read + end)."""
        out = np.empty((self.nbKangaroo, 12), dtype=np.uint64)
        self.WalksBegin()
        try:
            self.WalksRead(out.view(np.uint8).reshape(-1))
        finally:
            self.WalksEnd()
        return out

    def LoadWalks(self, recs, key=None, verify=True, bad_cap=None):
        """Write `recs` ((count, 12) uint64 or count * 96 uint8 records, count <= nbKangaroo) to kIdx [0, count); the rest
        of the herd is left as it is.  verify: check d*G (tame) / key + d*G (wild) for every record -> (n_bad, bad
        indices (ascending, at most bad_cap)); (0, empty) without verification."""
        a = np.ascontiguousarray(recs).view(np.uint8).reshape(-1)
        assert a.size % WALK_SIZE == 0
        count = a.size // WALK_SIZE
        if verify and key is None:
            raise ValueError("LoadWalks: verification needs the key")
        kx, ky = (_limbs([key[0]], 4), _limbs([key[1]], 4)) if key is not None else (np.zeros((1, 4), np.uint64), np.zeros((1, 4), np.uint64))
        cap = count if bad_cap is None else int(bad_cap)
        bad = np.zeros(max(cap, 1), dtype=np.uint64)
        nb = ctypes.c_uint64(0)
        self._ck(self._lib.kgx_walks_load(self._h, ctypes.c_void_p(a.ctypes.data), count, _p(self._wo()), _p(kx), _p(ky),
                                          int(bool(verify)), ctypes.byref(nb), _p(bad), ctypes.c_uint32(min(cap, 0xFFFFFFFF))), "LoadWalks")
        return int(nb.value), bad[:min(nb.value, cap)].copy()

    def callKernel(self):
        """GPUEngine.cu:540-557."""
        return self._lib.kgx_launch_async(self._h) == 0

    def Launch(self, spinWait=False, relaunch=True):
        """GPUEngine.cu:607-679: wait for the launch in flight, return its DPs (x, unbiased d, kIdx), start the
        next launch.  Returns the list (the reference fills `hashFound` and returns the launch status)."""
        n_items, n_found = ctypes.c_uint32(0), ctypes.c_uint32(0)
        self._ck(self._lib.kgx_collect(self._h, self._items, self.maxFound, ctypes.byref(n_items), ctypes.byref(n_found),
                                       int(bool(spinWait)), int(bool(relaunch))), "Launch")
        if n_found.value > self.maxFound and not self.lostWarning:
            print("\nWarning, %d items lost\nHint: Search with less threads (-g) or increse dp (-d)" %
                  (n_found.value - self.maxFound))
            self.lostWarning = True
        self.lastFound = n_found.value
        k = n_items.value
        if k == 0:
            return []
        # vectorised decode of the 56-byte records: 7 x u64 per item
        raw = np.frombuffer(self._items, dtype=np.uint64, count=k * 7).reshape(k, 7)
        xs = _ints(raw[:, 0:4]); ds = _ints(raw[:, 4:6]); ks = raw[:, 6].tolist()
        return [ITEM(x, self._unbias(d, kk), int(kk)) for x, d, kk in zip(xs, ds, ks)]

    def collect_count(self, spinWait=False, relaunch=True):
        """Launch() without the host copy of the records: wait for the launch in flight, (re)launch, return how many DPs it
        produced.  The records stay in the device slab (dp_slab_device_ptr / convert_dps_device_ptr) for the NCCL gather."""
        n_items, n_found = ctypes.c_uint32(0), ctypes.c_uint32(0)
        self._ck(self._lib.kgx_collect(self._h, self._items, 0, ctypes.byref(n_items), ctypes.byref(n_found),
                                       int(bool(spinWait)), int(bool(relaunch))), "Launch")
        self.lastFound = n_found.value
        return int(n_found.value)

    def callKernelAndWait(self):
        ok = self.callKernel()
        self._ck(self._lib.kgx_sync(self._h), "callKernelAndWait")
        return ok

    # -- extras (not in the reference class) ---------------------------------------------------------------
    def sync(self):
        self._ck(self._lib.kgx_sync(self._h), "sync")

    def last_launch_ms(self):
        return float(self._lib.kgx_last_launch_ms(self._h))

    def set_jumps_per_launch(self, n):
        self._ck(self._lib.kgx_set_jumps_per_launch(self._h, n), "set_jumps_per_launch")

    def kernel_launches(self):
        return int(self._lib.kgx_kernel_launches(self._h))

    def convert_dps_device_ptr(self):
        """HashTable::Convert on the device for the last completed launch -> device pointer of
        [u32 count][40-byte DP records] (Kangaroo.h:94-101)."""
        wo = _limbs([self.wildOffset & ((1 << 128) - 1)], 2)
        out = ctypes.c_void_p(0)
        self._ck(self._lib.kgx_convert_dps(self._h, _p(wo), ctypes.byref(out)), "convert_dps")
        return int(out.value)

    def dp_slab_device_ptr(self):
        return int(self._lib.kgx_dp_slab_device(self._h))


def random_herd_arrays(n, range_power, wdiv2, rng):
    """Vectorised distances for Kangaroo::CreateHerd (Kangaroo.cpp:696-704): v uniform in [0, 2^rangePower) for every
    kangaroo; tame scalar = v, wild scalar = v - width/2 (mod n).  Returns (scalars (n,4), d128 (n,2)) uint64 where d128
    is the device distance when wildOffset == width/2 (then wild bias + shift cancel: stored distance = v)."""
    assert range_power <= 128
    v = np.zeros((n, 4), dtype=np.uint64)
    for k in range((range_power + 63) // 64):
        v[:, k] = rng.integers(0, 1 << 63, size=n, dtype=np.uint64) * np.uint64(2) + rng.integers(0, 2, size=n, dtype=np.uint64)
    top = range_power % 64
    if top:
        v[:, (range_power - 1) // 64] &= np.uint64((1 << top) - 1)
    d128 = np.ascontiguousarray(v[:, :2])
    sc = v.copy()
    w = [(wdiv2 >> (64 * k)) & _M64 for k in range(4)]
    odd = np.arange(n) % 2 == WILD
    borrow = np.zeros(n, dtype=np.uint64)
    for k in range(4):                                   # sc[odd] -= wdiv2 (4-limb subtract with borrow)
        a = sc[:, k]
        sub = np.uint64(w[k])
        t = a - sub
        b1 = (a < sub).astype(np.uint64)
        t2 = t - borrow
        b2 = (t < borrow).astype(np.uint64)
        sc[:, k] = np.where(odd, t2, a)
        borrow = np.where(odd, b1 | b2, 0).astype(np.uint64)
    neg = borrow.astype(bool)                            # went negative: add the group order back
    carry = np.zeros(n, dtype=np.uint64)
    for k in range(4):
        a = sc[:, k]
        addv = np.uint64((ORDER >> (64 * k)) & _M64)
        t = a + addv
        c1 = (t < a).astype(np.uint64)
        t2 = t + carry
        c2 = (t2 < t).astype(np.uint64)
        sc[:, k] = np.where(neg, t2, a)
        carry = np.where(neg, c1 | c2, 0).astype(np.uint64)
    return sc, d128
