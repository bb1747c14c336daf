"""Stand-alone multi-GPU driver of the jump engine: the role Kangaroo::Run / SolveKeyGPU (Kangaroo.cpp:913-1083,
510-644) plays in the reference, with the reference's TCP client/server (Network.cpp) replaced in-box by one process
per GPU and an NCCL gather of the DP records to rank 0 (kangaroo_b200/dist.py).  Small on purpose -- it exists to run the
engine end to end at full multi-GPU speed (BASELINE config 4), and the full-featured caller remains the reference's own
program linked against the engine (INTEGRATION.md) -- except for checkpoints: a run of days must survive preemption, so it
writes and resumes the reference's work files, kangaroos included (-w / -wi / -ws / -i there, --work-file /
--work-interval / --save-kangaroos / --resume here).

Per step (= one GPUEngine::Launch on every rank) nothing on the data path is Python:
  engine      kgx_collect(cap=0, relaunch=1): wait for launch i, start launch i+1, no host copy of records
  device      kgx_convert_dps: HashTable::Convert of launch i's DPs -> 40-byte `DP` records (Kangaroo.h:94-101)
  NCCL        all_gather(count) + gather(records) to rank 0          (dist.DPGather, wire "dp40")
  rank 0      device table (dptable.DeviceDPTable, when it fits rank 0's memory): kgx_dpt_insert of the gathered buffer,
              stream-ordered, no host copy; its events are collected one step later
              host table otherwise: one D2H copy -> (ingest thread, one step behind, overlapping the next launch) kgi_add:
              the reference's HashTable, bucket-sharded multi-threaded insert (ingest.DPTable)
              -> events: KGI_EV_COLLISION -> kgi_resolve (CollisionCheck/CheckKey with the reference's Secp256K1)
                         KGI_EV_RESET     -> (rank, kIdx) sent back to the owner, which re-creates that kangaroo
                                             (Kangaroo.cpp:601-609: CreateHerd(1) + SetKangaroo)
  all ranks   one small broadcast: [stop, n_resets, checkpoint begin, checkpoint offset, (rank, kIdx) ...]

Checkpoints (kangaroo_b200/checkpoint.py for the file protocol).  The table in a checkpoint holds exactly the DPs of
launches 1..L, its walks are the herd after launch L on every rank and its count the jumps through launch L:
  step s      rank 0 decides, the control word carries "begin"; every rank calls kgx_walks_begin, which converts the
              herd on the device in stream order behind launch L = s + 1 (in flight) and returns at once
  step s + 1  launch L's records go to the table and rank 0 queues a save marker right behind them: the ingest thread
              writes header + table to F.tmp (the step loop stalls only if this outlasts the next step's insert); with the
              device table the marker is an export stream-ordered behind launch L's insert, which a thread of its own turns
              into F.tmp (kgi_fill_sorted + kgi_save_work_walks) while later inserts go on
  later       the walk offset goes out in a control word; every rank's writer thread copies its walks out in chunks and
              pwrites them; a MIN all-reduce of the ranks' done flags runs each step until all are written; rank 0 then
              fsyncs and renames F.tmp -> F
When the run stops without a key (--max-steps, SIGINT, SIGTERM) the launch in flight is collected too and a last
checkpoint is written the same way, synchronously.

  single GPU :  python -m kangaroo_b200.solver in.txt --dp 12
  N GPUs     :  torchrun --nproc-per-node N -m kangaroo_b200.solver in.txt --dp 12
  checkpoint :  ... --work-file run.work --work-interval 600 --save-kangaroos
  resume     :  python -m kangaroo_b200.solver --resume run.work [--work-file run.work ...]
"""
import argparse
import ctypes
import os
import queue
import signal
import sys
import threading
import time

import numpy as np

from . import ecmath as ec
from . import checkpoint as ckpt
from .engine import GPUEngine, NB_JUMP, NB_RUN, WILD, WALK_SIZE, random_herd_arrays
from .dist import DPGather, SlabView, DP40_BYTES
from .ingest import DPTable, EV_RESET, EV_COLLISION, read_work_info
from . import dptable

ORDER = ec.N
MAX_RESETS = 255          # per step, carried in the control broadcast
CTRL_HEAD = 4             # control word: stop, n_resets, checkpoint begin, checkpoint walk offset (-1: table write failed)
STOP_KEY, STOP_SIGNAL = 1, 2
WALK_CHUNK = 1 << 18      # walks per pinned chunk of a checkpoint writer (24 MiB)

_signalled = []           # SIGINT / SIGTERM received (main() installs the handler)


def _on_signal(signum, frame):
    _signalled.append(signum)


class _Checkpoint:
    """One checkpoint in progress on this rank."""

    def __init__(self, path, final):
        self.path, self.final = path, final
        self.phase = "exported"          # -> "table" (marker queued, rank 0) -> "writing" (offset known)
        self.t0 = time.time()
        self.result = queue.Queue()      # rank 0: walk offset from the ingest thread (or an exception)
        self.writer = None
        self.stall0 = 0.0


def create_jump_table(range_power):
    """Kangaroo::CreateJumpTable (Kangaroo.cpp:742-832, non-symmetry): 32 distances of rangePower/2+1 bits from MT19937
    seeded 0x600DCAFE (constant "for compatibility of workfiles"), redrawn until the mean is within 2^(jumpBit-1.05 ..
    -0.95); points = d*G.  numpy's RandomState is the same MT19937 with the same seeding, Int::Rand(nbit) consumes
    nbit/32 + 1 words (Int.cpp:988-1001)."""
    jump_bit = min(range_power // 2 + 1, 128)
    rs = np.random.RandomState(0x600DCAFE)
    lo, hi = 2.0 ** (jump_bit - 1.05), 2.0 ** (jump_bit - 0.95)
    nb, left = jump_bit // 32, jump_bit % 32
    for _ in range(100):
        dist = []
        for _i in range(NB_JUMP):
            words = [int(v) for v in rs.randint(0, 2**32, size=nb + 1, dtype=np.uint64)]
            words[nb] &= (1 << left) - 1
            v = sum(w << (32 * k) for k, w in enumerate(words))
            dist.append(v or 1)
        if lo < sum(dist) / NB_JUMP < hi:
            break
    pts = [ec.mul(d) for d in dist]
    return dist, [p[0] for p in pts], [p[1] for p in pts]


def dp_mask(bits):
    """Kangaroo::SetDP (Kangaroo.cpp:154-164)"""
    return 0 if bits == 0 else (~((1 << (64 - min(bits, 64))) - 1)) & 0xFFFFFFFFFFFFFFFF


class Solver:
    def __init__(self, start, end, pub, dp_bits, grid=None, max_found=1 << 17, seed=None, ingest_threads=0,
                 work_file="", work_interval=0.0, save_kangaroos=False, resume=None):
        import torch
        self.torch = torch
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(self.local)
        self.dist = None
        if self.world > 1:
            import torch.distributed as dist
            if not dist.is_initialized():
                dist.init_process_group("nccl", device_id=torch.device("cuda", self.local))
            self.dist = dist
        self.start, self.end, self.pub, self.dp_bits = start, end, pub, dp_bits
        width = end - start
        self.range_power = width.bit_length()                         # Kangaroo::InitRange (:877-890)
        self.wdiv2 = width >> 1
        # Kangaroo::InitSearchKey (:892-909): keyToSearch = P - start*G
        self.key = ec.add(pub, ec.neg(ec.mul(start))) if start else pub
        gx, gy = grid or GPUEngine.GetGridSize(self.local, 0, 0)
        self.eng = GPUEngine(gx, gy, self.local, max_found)
        self.table = create_jump_table(self.range_power)
        self.eng.SetParams(dp_mask(dp_bits), *self.table)
        self.eng.SetWildOffset(self.wdiv2)
        # Kangaroo::CreateHerd (:670-738): tame d in [0, 2^rangePower), wild d - width/2; points on the device
        n = self.eng.nbKangaroo
        self.rng = np.random.Generator(np.random.PCG64((seed if seed is not None else int(time.time())) * 1000 + self.rank))
        sc, d128 = random_herd_arrays(n, self.range_power, self.wdiv2, self.rng)
        self.eng.CreateHerdRaw(sc, d128, self.key)
        self.gather = DPGather(self.eng, self.dist, self.rank, self.world, torch, wire="dp40") if self.world > 1 else None
        self.dps = DPTable(threads=ingest_threads) if self.rank == 0 else None      # rank 0: the reference HashTable
        self.dev = None                     # rank 0: the device table, when chosen (_choose_table)
        self.table_kind = "host"
        self._lost_warned = False
        self.work_file, self.work_interval, self.save_kangaroos = work_file, float(work_interval or 0), bool(save_kangaroos)
        self.jumps0, self.time0 = 0, 0.0
        self.loaded = self.bad = 0
        # Two pinned staging buffers: while the ingest thread inserts step k's records, step k+1's land in the other one.  The
        # NCCL kernels of a step cannot start before the jump launch that occupies every SM has finished, so without this
        # decoupling the CPU insert (3-4 ms at 8 GPUs) sat exposed between two launches: 97 instead of 112 GJump/s.
        self._hosts = None                  # allocated on the first host-table step
        self._max_found = max_found
        self._dpbuf = None                  # single GPU, device table: this step's records, off the engine's buffer
        self._ck_table = None               # device table: host table a checkpoint is written from
        self._hidx = 0
        self._work = queue.Queue()          # steps' records (at most two in flight, _staging) and checkpoint markers
        self._done = queue.Queue()
        self._pending = 0
        self._acc_found, self._acc_resets = None, []
        self._thread = None
        if self.rank == 0:
            self._thread = threading.Thread(target=self._ingest_loop, daemon=True)
            self._thread.start()
        self._ctrl = torch.zeros(CTRL_HEAD + 2 * MAX_RESETS, dtype=torch.int64, device="cuda")
        self._flag = torch.zeros(1, dtype=torch.int64, device="cuda")
        self.jumps = self.jumps0
        self.stop_reason = 0
        self._ck = None
        self._ck_last = time.time()
        self._ck_host = None
        self.t_stall = 0.0                  # step loop blocked by checkpoints: export set-up + waits behind the table write
        self._table_busy = False            # ingest thread is writing a checkpoint's header and table
        self.checkpoints = []               # rank 0: (path, bytes, seconds, stall seconds) of every committed checkpoint
        self.same_herd = 0
        self.resets_done = 0
        self.t_ingest = 0.0
        self.stop = False
        if resume:
            self._resume(resume, n)
            self.jumps = self.jumps0
        self.expected_ops = dptable.compute_expected(self.range_power, n * self.world, dp_bits)[0]
        self.suggested_dp = dptable.suggested_dp(self.range_power, n * self.world)
        if self.rank == 0:
            self._choose_table()

    def _choose_table(self):
        """rank 0: the device table when 2 E entries (at least 1.5 E) fit 3/4 of the free device memory, E = the expected DP
        count plus the resumed entries; KGX_DPTABLE / KGX_DPTABLE_CAP pin the choice"""
        loaded = len(self.dps)
        self.expected_dps = self.expected_ops / 2.0 ** self.dp_bits + loaded
        free = self.torch.cuda.mem_get_info(self.local)[0]
        kind, cap = dptable.choose_from_env(self.expected_dps, free)
        if kind == "device" and loaded > cap:
            kind = "host"
        if kind == "device":
            self.dev = dptable.DeviceDPTable(self.local, cap)
            if loaded:
                self.dev.load_from_host(self.dps)
                self.dps.reset()
        self.table_kind = kind

    def table_len(self):
        return self.dev.entries if self.dev is not None else len(self.dps)

    def table_desc(self):
        if self.dev is None:
            return "host (%d ingest threads)" % self.dps.threads
        return "device (%d entries, %.1f GB)" % (self.dev.capacity, self.dev.memory() / 1e9)

    # -- rank 0: ingest -------------------------------------------------------------------------------------------
    def _events(self, events, found, resets):
        for kind, rk, kidx, d_old, d_new in events:
            if kind == EV_COLLISION and found is None:
                found = self.dps.resolve(d_old, d_new, self.key, self.start)     # Kangaroo.cpp:255-302
                if found is None:
                    resets.append((rk, kidx))                                    # "unexpected wrong collision, reset kangaroo"
            elif kind == EV_RESET:
                resets.append((rk, kidx))
        return found

    def _ingest(self, segments):
        """segments: list of (rank, uint8 numpy view of that rank's 40-byte records).  Returns (key or None, resets)."""
        found, resets = None, []
        t0 = time.perf_counter()
        for r, buf in segments:
            if buf.size == 0:
                continue
            found = self._events(self.dps.add_dp40(buf, r), found, resets)
        self.t_ingest += time.perf_counter() - t0
        return found, resets

    def _ingest_loop(self):
        while True:
            segs = self._work.get()
            if segs is None:
                return
            if isinstance(segs, _Checkpoint):
                self._write_table(segs)
                continue
            self._done.put(self._ingest(segs))

    def _write_table(self, ck):
        """ingest thread, at the save marker: every DP of launches 1..L is in the table, none of a later launch"""
        self._table_busy = True
        try:
            walks = self.eng.nbKangaroo * self.world if self.save_kangaroos else 0
            off = self.dps.save_work_walks(ckpt.tmp_path(ck.path), self.dp_bits, self.start, self.end, self.pub,
                                           total_count=ck.count, total_time=ck.time, total_walks=walks)
            ck.result.put(off)
        except BaseException as e:
            ck.result.put(e)
        finally:
            self._table_busy = False

    def _submit(self, segs):
        """hand one step's records to the ingest thread"""
        self._work.put(segs)
        self._pending += 1

    def _staging(self):
        """the staging buffer for this step; at most one older step may still be in the ingest thread (it reads the OTHER buffer)"""
        t0 = time.perf_counter() if self._table_busy else None   # only a wait that starts behind a table write is its cost
        while self._pending >= 2:
            self._take(block=True)
        if t0 is not None:
            self.t_stall += time.perf_counter() - t0
        if self._hosts is None:
            self._hosts = [self.torch.empty(self.world * self._max_found * DP40_BYTES, dtype=self.torch.uint8).pin_memory() for _ in range(2)]
        host = self._hosts[self._hidx]
        self._hidx ^= 1
        return host

    def _take(self, block):
        f, r = self._done.get(block=block)
        self._pending -= 1
        if self._acc_found is None:
            self._acc_found = f
        self._acc_resets += r

    def _take_dev(self):
        """events of the oldest insert queued on the device table"""
        t0 = time.perf_counter()
        resets = []
        f = self._events(self.dev.events(), None, resets)
        self.t_ingest += time.perf_counter() - t0
        if self._acc_found is None:
            self._acc_found = f
        self._acc_resets += resets

    def _dev_insert(self, ptr, counts, stride):
        """rank 0: one step's records (device memory) into the device table; False when they would take it past its
        capacity (the caller then migrates and uses the host table)"""
        n = sum(counts)
        if not self.dev.fits(n):
            while self.dev.pending:                                     # the exact count, then decide
                self._take_dev()
            if not self.dev.fits(n):
                return False
        while self.dev.pending >= 2:
            self._take_dev()
        t0 = time.perf_counter()
        self.dev.insert(ptr, counts, stride, self.torch.cuda.current_stream().cuda_stream)
        self.t_ingest += time.perf_counter() - t0
        return True

    def _migrate(self):
        """rank 0: the device table is full -- move its content to the host table once and go on there"""
        t0 = time.perf_counter()
        ck = self._ck
        if ck is not None and ck.phase == "table" and getattr(ck, "thread", None) is not None:
            ck.thread.join()                                            # its export reads the device table
        while self.dev.pending:
            self._take_dev()
        n = self.dev.entries
        self.dev.to_host(self.dps, self.torch.cuda.current_stream().cuda_stream)
        cap = self.dev.capacity
        self.dev.close()
        self.dev = None
        self.table_kind = "host"
        self.t_stall += time.perf_counter() - t0
        print("DP table: the device table is full (%d of %d entries), moved to the host table in %.2f s; the run goes on there" %
              (n, cap, time.perf_counter() - t0), flush=True)

    def _harvest(self, wait_all=False):
        """results of the inserts finished so far -> (key or None, resets)"""
        if self.dev is not None:
            while self.dev.pending > (0 if wait_all else 1):            # one step behind: the newest insert may still run
                self._take_dev()
        while self._pending and (wait_all or not self._done.empty()):
            self._take(block=True)
        found, resets = self._acc_found, self._acc_resets
        self._acc_found, self._acc_resets = None, []
        return found, resets

    def _reset_kangaroo(self, kidx):
        """Kangaroo.cpp:601-609: CreateHerd(1, type) + SetKangaroo(kIdx) on the owning engine."""
        v = int(self.rng.integers(0, 1 << 62)) | (int(self.rng.integers(0, 1 << 62)) << 62) | (int(self.rng.integers(0, 1 << 62)) << 124)
        v &= (1 << self.range_power) - 1
        if kidx % 2 == WILD:
            d = (v - self.wdiv2) % ORDER
            pos = ec.add(self.key, ec.mul(d))
        else:
            d = v
            pos = ec.mul(d)
        if pos is None:
            return
        self.eng.SetKangaroo(kidx, pos[0], pos[1], d)
        self.resets_done += 1

    def step(self, relaunch=True):
        """one Launch on every rank; returns the private key on rank 0 when found (None otherwise).  relaunch=False
        collects the launch in flight without starting another (the last step before a final checkpoint)."""
        torch = self.torch
        n_found = self.eng.collect_count(relaunch=relaunch)              # launch i done, launch i+1 running
        cnt = min(n_found, self.eng.maxFound)
        if n_found > cnt and not self._lost_warned:                       # GPUEngine.cu:641-648
            print("\nWarning, %d items lost (rank %d)\nHint: Search with less threads (-g) or increse dp (-d)" %
                  (n_found - cnt, self.rank), flush=True)
            self._lost_warned = True
        self.jumps += self.eng.nbKangaroo * NB_RUN * self.world
        found, resets = None, []
        if self.gather is not None:
            res = self.gather.step_flat(cnt)                                # rank 0: (counts, cap, device tensor [world*cap*40])
            if self.rank == 0 and self.dev is not None and self._dev_insert(res[2].data_ptr(), res[0], res[1]):
                pass
            elif self.rank == 0:
                if self.dev is not None:
                    self._migrate()
                counts, cap, flat = res
                nbytes = self.world * cap * DP40_BYTES
                host = self._staging()
                host[:nbytes].copy_(flat[:nbytes], non_blocking=True)
                torch.cuda.current_stream().synchronize()
                h = host.numpy()
                self._submit([(r, h[r * cap * DP40_BYTES: r * cap * DP40_BYTES + counts[r] * DP40_BYTES]) for r in range(self.world)])
        else:
            if cnt:
                ptr = self.eng.convert_dps_device_ptr()
                dev = torch.as_tensor(SlabView(ptr + 4, cnt * DP40_BYTES), device="cuda")
                if self.dev is not None:
                    # the engine rewrites its buffer at the next step: the insert reads a copy, ordered before it on this stream
                    if self._dpbuf is None:
                        self._dpbuf = torch.empty(self._max_found * DP40_BYTES, dtype=torch.uint8, device="cuda")
                    self._dpbuf[:cnt * DP40_BYTES].copy_(dev)
                    ev = torch.cuda.Event()
                    ev.record()
                    if self._dev_insert(self._dpbuf.data_ptr(), [cnt], 0):
                        ev.synchronize()
                        cnt = 0
                    else:
                        self._migrate()
            if cnt:
                host = self._staging()
                host[:cnt * DP40_BYTES].copy_(dev, non_blocking=True)
                torch.cuda.current_stream().synchronize()
                self._submit([(0, host.numpy()[:cnt * DP40_BYTES])])
        ck_begin, ck_off = 0, 0
        if self.rank == 0:
            self._ck_marker()                                               # right behind launch L's records
            found, resets = self._harvest()
            stop = STOP_KEY if found is not None else (STOP_SIGNAL if _signalled else 0)
            if (self._ck is None and self.work_file and self.work_interval > 0 and not stop and relaunch
                    and time.time() - self._ck_last >= self.work_interval):
                ck_begin = 1
            ck_off = self._ck_offset(block=False)
        # control word: stop flag, checkpoint, kangaroos to re-create, back to their owners
        if self.dist is not None:
            if self.rank == 0:
                resets = resets[:MAX_RESETS]
                c = [stop, len(resets), ck_begin, ck_off] + [v for rk in resets for v in rk]
                self._ctrl[:len(c)].copy_(torch.tensor(c, dtype=torch.int64))
            self.dist.broadcast(self._ctrl, 0)
            c = self._ctrl[:CTRL_HEAD + 2 * MAX_RESETS].cpu().tolist()
            stop, ck_begin, ck_off = c[0], c[2], c[3]
            resets = [(c[CTRL_HEAD + 2 * i], c[CTRL_HEAD + 1 + 2 * i]) for i in range(c[1])]
        self.stop_reason = stop
        self.stop = bool(stop)
        if ck_begin:
            self._ck_begin(final=False)
        if ck_off:
            self._ck_write(ck_off)
        if self._ck is not None and self._ck.phase == "writing":
            self._ck_poll_done(block=False)
        # A kangaroo reset below was exported by a checkpoint begun in this step as it was before the reset: on resume it
        # re-emits a DP the table already holds and is reset again -- harmless.
        for rk, kidx in resets:
            self.same_herd += 1
            if rk == self.rank and not self.stop:
                self._reset_kangaroo(kidx)
        return found

    # -- checkpoints ------------------------------------------------------------------------------------------------
    def _ck_begin(self, final):
        """every rank, in the same step: export the herd behind the launch in flight (or, final, the last launch)"""
        t0 = time.perf_counter()
        self._ck = _Checkpoint(self.work_file, final)
        self._ck.stall0 = self.t_stall
        if self.save_kangaroos:
            self.eng.WalksBegin()
        self.t_stall += time.perf_counter() - t0

    def _ck_marker(self):
        """rank 0, after submitting the records of launch L: queue the table write behind them"""
        ck = self._ck
        if ck is None or ck.phase != "exported":
            return
        ck.count = self.jumps
        ck.time = self.time0 + (time.time() - self._t_run)
        ck.phase = "table"
        if self.dev is not None:
            self.dev.export_begin(self.torch.cuda.current_stream().cuda_stream)   # behind launch L's insert
            ck.thread = threading.Thread(target=self._write_table_dev, args=(ck,), daemon=True)
            ck.thread.start()
        else:
            self._work.put(ck)

    def _write_table_dev(self, ck):
        """thread of its own, device table: the export of launches 1..L -> a host table in work-file order -> F.tmp"""
        try:
            if self._ck_table is None:
                self._ck_table = DPTable(threads=1)
            self.dev.export_to_host(self._ck_table)
            walks = self.eng.nbKangaroo * self.world if self.save_kangaroos else 0
            off = self._ck_table.save_work_walks(ckpt.tmp_path(ck.path), self.dp_bits, self.start, self.end, self.pub,
                                                 total_count=ck.count, total_time=ck.time, total_walks=walks)
            ck.result.put(off)
        except BaseException as e:
            ck.result.put(e)
        finally:
            if self._ck_table is not None:
                self._ck_table.reset()                                  # the host copy is not kept between checkpoints

    def _ck_offset(self, block):
        """rank 0: the walk offset once the ingest thread wrote header and table (0 while pending, -1 on failure)"""
        ck = self._ck
        if ck is None or ck.phase != "table" or getattr(ck, "offset", None) is not None:
            return 0
        try:
            r = ck.result.get(block=block)
        except queue.Empty:
            return 0
        if isinstance(r, BaseException):
            print("checkpoint: cannot write %s: %s" % (ckpt.tmp_path(ck.path), r), flush=True)
            r = -1
        ck.offset = r
        return r

    def _ck_write(self, offset):
        """every rank: start writing this rank's walks at the offset rank 0 announced"""
        ck = self._ck
        ck.phase = "writing"
        if offset < 0:
            ck.failed = True
            return
        if not self.save_kangaroos:
            return
        n = self.eng.nbKangaroo
        if self._ck_host is None:
            self._ck_host = self.torch.empty(min(WALK_CHUNK, n) * WALK_SIZE, dtype=self.torch.uint8).pin_memory()
        host = self._ck_host
        eng = self.eng

        def read(buf, first, count):
            eng.WalksRead(host, first, count)
        ck.writer = ckpt.SliceWriter(ckpt.tmp_path(ck.path), offset, self.rank * n, n, read, host.numpy(), min(WALK_CHUNK, n),
                                     on_exit=eng.WalksEnd)

    def _ck_local_state(self):
        ck = self._ck
        if getattr(ck, "failed", False):
            return -1
        return ck.writer.state if ck.writer is not None else 1

    def _ck_poll_done(self, block):
        """every rank, in the same step: have all ranks written their walks?  rank 0 then commits the file"""
        ck = self._ck
        if block and ck.writer is not None:
            ck.writer.join()
        st = self._ck_local_state()
        if self.dist is not None:
            self._flag.fill_(st)
            self.dist.all_reduce(self._flag, op=self.dist.ReduceOp.MIN)
            st = int(self._flag.item())
        if st == 0:
            return
        self._ck_release(ck)
        if self.rank == 0:
            if st == 1:
                ckpt.commit(ck.path)
                size = os.path.getsize(ck.path)
                dt, stall = time.time() - ck.t0, self.t_stall - ck.stall0
                self.checkpoints.append((ck.path, size, dt, stall))
                print("checkpoint: %s  %.1f MB  %.2f s  (step loop waited %.3f s)" % (ck.path, size / 1e6, dt, stall), flush=True)
            else:
                ckpt.discard(ck.path)
                print("checkpoint: %s not written, the previous file is kept" % ck.path, flush=True)
        self._ck = None
        self._ck_last = time.time()

    def _ck_release(self, ck):
        """this rank's side of a checkpoint that is over: writer joined, export ended (also when no writer ran, e.g. after a
        failed table write), so the next checkpoint can begin"""
        if getattr(ck, "thread", None) is not None:
            ck.thread.join()
        if ck.writer is not None:
            ck.writer.join()
            if ck.writer.error is not None:
                print("checkpoint: rank %d could not write its walks: %s" % (self.rank, ck.writer.error), flush=True)
        elif self.save_kangaroos:
            self.eng.WalksEnd()

    def _ck_abandon(self):
        """the run ends with a checkpoint in progress (the key was found): finish what is running on this rank -- the walk
        writer, the table write queued on rank 0 -- before the engine and the table go away, and drop F.tmp.  Local only:
        no collective, every rank does the same."""
        ck = self._ck
        if ck is None:
            return
        self._ck_release(ck)
        if self.rank == 0:
            if ck.phase == "table" and getattr(ck, "offset", None) is None:
                ck.result.get()                             # the ingest thread is writing or about to write the table
            ckpt.discard(ck.path)
            print("checkpoint: %s abandoned, the run ended while it was written; the previous file is kept" % ck.path, flush=True)
        self._ck = None

    def _ck_finish(self):
        """every rank: drive the checkpoint in progress to its end, blocking"""
        ck = self._ck
        if ck is None:
            return
        if self.rank == 0:
            self._ck_marker()
        if ck.phase != "writing":
            off = self._ck_offset(block=True) if self.rank == 0 else 0
            if self.dist is not None:
                self._flag.fill_(off)
                self.dist.broadcast(self._flag, 0)
                off = int(self._flag.item())
            self._ck_write(off)
        self._ck_poll_done(block=True)

    def final_checkpoint(self):
        """the run stopped without a key: collect the launch in flight, then write a checkpoint of the state after it"""
        key = self.step(relaunch=False)
        if self.stop_reason == STOP_KEY:
            return key
        self._ck_finish()                                   # a periodic checkpoint still in progress
        self._ck_begin(final=True)
        self._ck_finish()
        return None

    # -- resume -----------------------------------------------------------------------------------------------------
    def _resume(self, path, n):
        """Kangaroo::LoadWork + FectchKangaroos (Backup.cpp:154-200, 291-359): rank 0 takes the table, every rank its slice
        of the walks; the herd created above keeps the kangaroos the file lacks."""
        info = read_work_info(path, self.dps)          # rank 0 loads the table, the other ranks skip it
        self.jumps0, self.time0 = info.total_count, info.total_time
        first = self.rank * n
        count = max(0, min(n, info.n_walks - first))
        err = None
        try:
            if count:
                err = self._load_slice(info, first, count, n)
            elif self.rank == 0:
                print("resume: no walks in %s, %d kangaroos created fresh per GPU" % (info.path, n), flush=True)
        except Exception as e:                              # e.g. an unreadable file, a failed device call
            err = "resume: rank %d: %s" % (self.rank, e)
        if self.dist is not None:                           # every rank stops when one cannot go on, none waits in a collective
            self._flag.fill_(0 if err else 1)
            self.dist.all_reduce(self._flag, op=self.dist.ReduceOp.MIN)
            if not err and int(self._flag.item()) == 0:
                err = "resume: rank %d: another rank could not resume from %s" % (self.rank, info.path)
        if err:
            raise SystemExit(err)
        left = info.n_walks - self.world * n
        if self.rank == 0 and left > 0:
            print("FectchKangaroos: Warning %d unhandled kangaroos !" % left, flush=True)

    def _load_slice(self, info, first, count, n):
        """this rank's walks [first, first + count) of the file into kIdx [0, count), checked; -> error text or None"""
        recs = np.fromfile(info.path, dtype=np.uint8, count=count * WALK_SIZE, offset=info.walk_offset + first * WALK_SIZE)
        if recs.size != count * WALK_SIZE:
            return "resume: %s is truncated (walks of rank %d missing)" % (info.path, self.rank)
        t0 = time.time()
        nbad, bad = self.eng.LoadWalks(recs, key=self.key, verify=True)
        # tame walks (d*G) are valid for any key: a file of another key fails on the wild half only
        bad_wild = int(np.count_nonzero(bad & 1))
        if 2 * nbad > count or 2 * bad_wild > count // 2:
            return ("resume: %d of %d walks (%d wild) of %s fail d*G (+key) = position: the file does not belong to this key "
                    "and range" % (nbad, count, bad_wild, info.path))
        for kidx in bad:
            self._reset_kangaroo(int(kidx))
        self.loaded, self.bad = count, nbad
        print("resume: rank %d: %d walks loaded and checked in %.2f s, %d re-created, %d created fresh" %
              (self.rank, count, time.time() - t0, nbad, n - count), flush=True)
        return None

    def run(self, max_steps=1 << 30, verbose=True):
        self.eng.callKernel()
        t0 = time.time()
        self._t_run = t0
        self._ck_last = t0
        key = None
        steps = 0
        self.steady = None                      # (time, jumps) after the first 32 steps: NCCL communicator set-up, first table growth
        for s in range(max_steps):
            key = self.step()
            steps += 1
            if steps == 32:
                self.steady = (time.time(), self.jumps)
            if verbose and self.rank == 0 and (s % 64 == 63 or self.stop):
                dt = time.time() - t0
                print("[%6.1fs] 2^%.2f jumps  %.0f MJump/s  %d DPs  dead %d  ingest %.1f ms/step" %
                      (self.time0 + dt, np.log2(max(self.jumps, 1)), (self.jumps - self.jumps0) / dt / 1e6, self.table_len(),
                       self.same_herd, 1e3 * self.t_ingest / steps), flush=True)
            if self.stop:
                break
        t_loop, jumps_loop = time.time(), self.jumps           # the steady rate leaves the last checkpoint out
        if self.work_file and self.stop_reason != STOP_KEY:
            k = self.final_checkpoint()
            steps += 1
            key = key if key is not None else k
        self._ck_abandon()
        self.eng.sync()
        if self.rank == 0 and key is None:                      # the last steps' records may still be in the ingest thread
            key, _ = self._harvest(wait_all=True)
        t1 = time.time()
        self.elapsed = t1 - t0
        self.steps = steps
        self.steady_rate = ((jumps_loop - self.steady[1]) / (t_loop - self.steady[0]) if self.steady and steps > 64
                            else (self.jumps - self.jumps0) / self.elapsed)
        return key

    def close(self):
        self._ck_abandon()
        if self._thread is not None:
            self._harvest(wait_all=True)
            self._work.put(None)
            self._thread.join(timeout=10)
            self._thread = None
        if self.dev is not None:
            while self.dev.pending:
                self.dev.events()
            self.dev.close()
            self.dev = None
        self.eng.close()
        if self.dps is not None:
            self.dps.close()
        if self._ck_table is not None:
            self._ck_table.close()


def main(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("config", nargs="?", default=None, help="range start, range end, public keys (not needed with --resume)")
    ap.add_argument("--dp", type=int, default=None, help="distinguished-point bits (default 12, or the resumed file's)")
    ap.add_argument("--grid", default="")
    ap.add_argument("--seed", type=int, default=None)
    ap.add_argument("--max-steps", type=int, default=1 << 30)
    ap.add_argument("--ingest-threads", type=int, default=0, help="workers of the rank-0 DP table (0 = min(8, cores))")
    ap.add_argument("--save-work", default="", help="write the rank-0 DP table as a reference work file (HEADW) at the end")
    ap.add_argument("--work-file", default="", help="write checkpoints (reference work files) to this file (reference -w)")
    ap.add_argument("--work-interval", type=float, default=0.0,
                    help="seconds between checkpoints (reference -wi); without it a checkpoint is written only when the run "
                         "stops without the key (--max-steps, SIGINT, SIGTERM)")
    ap.add_argument("--save-kangaroos", action="store_true", help="checkpoints include every rank's kangaroos (reference -ws)")
    ap.add_argument("--resume", default="", help="continue from this work file: range, key, dp, count and time (reference -i)")
    a = ap.parse_args(argv)
    if a.resume:
        info = read_work_info(a.resume)
        start, end, pubs = info.range_start, info.range_end, [info.key]
        dp = a.dp if a.dp is not None else info.dp_bits
    elif a.config:
        start, end, pubs = ec.parse_config(a.config)
        dp = a.dp if a.dp is not None else 12
    else:
        ap.error("a config file or --resume is required")
    if (a.work_interval or a.save_kangaroos) and not a.work_file:
        ap.error("--work-interval and --save-kangaroos need --work-file")
    grid = tuple(int(v) for v in a.grid.split(",")) if a.grid else None
    if a.work_file:
        for sig in (signal.SIGINT, signal.SIGTERM):       # stop at the next step and write a last checkpoint
            signal.signal(sig, _on_signal)
    rc = 0
    for i, pub in enumerate(pubs):
        s = Solver(start, end, pub, dp, grid, seed=a.seed, ingest_threads=a.ingest_threads, work_file=a.work_file,
                   work_interval=a.work_interval, save_kangaroos=a.save_kangaroos, resume=a.resume or None)
        if s.rank == 0:
            print("Suggested DP: %d" % s.suggested_dp)
            print("Expected operations: 2^%.2f" % np.log2(s.expected_ops))
            print("Range width: 2^%d  kangaroos/GPU: %d  GPUs: %d  dp: %d  DP table: %s" %
                  (s.range_power, s.eng.nbKangaroo, s.world, dp, s.table_desc()), flush=True)
            if a.resume:
                print("resume: %s  count 2^%.2f  time %.1f s" % (a.resume, np.log2(max(s.jumps0, 1)), s.time0), flush=True)
        key = s.run(a.max_steps)
        if s.rank == 0:
            print("Solver rate: %.0f MJump/s steady state (after the first 32 steps), %.0f MJump/s over all %d steps (%.2f s); "
                  "rank-0 ingest %.2f ms/step; %d DPs; %d dead kangaroos re-created" %
                  (s.steady_rate / 1e6, (s.jumps - s.jumps0) / s.elapsed / 1e6, s.steps, s.elapsed, 1e3 * s.t_ingest / max(s.steps, 1),
                   s.table_len(), s.same_herd))
            print("Total count: %d jumps (2^%.2f)" % (s.jumps, np.log2(max(s.jumps, 1))))
            if a.save_work:
                if s.dev is not None:
                    s.dev.to_host(s.dps, s.torch.cuda.current_stream().cuda_stream)
                s.dps.save_work(a.save_work, dp, start, end, pub, total_count=s.jumps, total_time=s.time0 + s.elapsed)
                print("work file written: %s" % a.save_work)
            if key is not None and ec.mul(key) == pub:
                print("Key#%2d Pub:  0x%064X\n       Priv: 0x%X" % (i, pub[0], key))
            else:
                print("Key#%2d not found" % i); rc = 1
        s.close()
        if _signalled:
            break
    try:
        import torch.distributed as dist
        if dist.is_initialized():
            dist.destroy_process_group()
    except Exception:
        pass
    return rc


if __name__ == "__main__":
    sys.exit(main())
