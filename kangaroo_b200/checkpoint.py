"""Checkpoint files of the solver: reference work files (HEADW) that carry the kangaroos, written by several processes.

A checkpoint of F is built in F.tmp and renamed over F only once it is complete, so an interruption at any point leaves
the previous F as it was:

  rank 0        DPTable.save_work_walks(F.tmp, ..., total_walks=world * n): header + DP table + walk count; the file is
                extended to its final size, and the byte offset of the first walk record is handed to every rank
  every rank    write_slice(): its own walks -- kangaroos [rank * n, (rank + 1) * n) of the file -- in chunks, pwrite at
                offset + rank * n * 96, from a thread of its own
  rank 0        once every rank reported its slice written: commit() = fsync, rename F.tmp -> F, fsync the directory

All ranks run on one host (the solver's in-box multi-GPU mode), so F.tmp is the same file for all of them.
"""
import os
import threading
import time

WALK_BYTES = 96


def tmp_path(path):
    return path + ".tmp"


def write_slice(tmp, offset, first_walk, count, read, buf, chunk):
    """pwrite walks [first_walk, first_walk + count) of the file.  read(buf, i, k) fills buf with records [i, i + k) of
    this writer's slice (i relative to the slice); buf holds chunk records.  Returns the bytes written."""
    fd = os.open(tmp, os.O_WRONLY)
    try:
        done = 0
        while done < count:
            k = min(chunk, count - done)
            read(buf, done, k)
            view = memoryview(buf).cast("B")[:k * WALK_BYTES]
            pos = offset + (first_walk + done) * WALK_BYTES
            while len(view):
                w = os.pwrite(fd, view, pos)
                view, pos = view[w:], pos + w
            done += k
        return count * WALK_BYTES
    finally:
        os.close(fd)


def commit(path):
    """Make F.tmp durable and put it in place of F."""
    tmp = tmp_path(path)
    fd = os.open(tmp, os.O_RDONLY)
    try:
        os.fsync(fd)
    finally:
        os.close(fd)
    os.replace(tmp, path)
    dfd = os.open(os.path.dirname(os.path.abspath(path)), os.O_RDONLY)
    try:
        os.fsync(dfd)
    finally:
        os.close(dfd)


def discard(path):
    try:
        os.unlink(tmp_path(path))
    except OSError:                         # absent, or not removable: F itself is untouched either way
        pass


class SliceWriter:
    """One rank's walk slice written from a background thread.  state: 0 running, 1 written, -1 failed (error kept)."""

    def __init__(self, tmp, offset, first_walk, count, read, buf, chunk, on_exit=None):
        self.state, self.error, self.seconds = 0, None, 0.0
        self._args = (tmp, offset, first_walk, count, read, buf, chunk)
        self._on_exit = on_exit
        self._thread = threading.Thread(target=self._run, daemon=True)
        self._thread.start()

    def _run(self):
        t0 = time.perf_counter()
        st = 1
        try:
            write_slice(*self._args)
        except BaseException as e:          # reported through the done flag; rank 0 then drops F.tmp
            self.error, st = e, -1
        if self._on_exit is not None:
            try:
                self._on_exit()
            except BaseException as e:
                if self.error is None:
                    self.error, st = e, -1
        self.seconds = time.perf_counter() - t0
        self.state = st                     # last: the caller may start the next export once it reads 1 or -1

    def join(self):
        self._thread.join()
        return self.state
