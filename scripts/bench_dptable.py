"""Device vs host DP table: insert throughput and checkpoint export time at given table sizes, and optionally the solver's
steady rate at two dp values on both tables.  Prints one JSON object per measurement, card name and power limit first.

  python scripts/bench_dptable.py --sizes 1e7,1e8,6e8 --batches 38000,606000
  python scripts/bench_dptable.py --sizes 0 --solver --gpus 8 --dps 16,12 --max-steps 600

Tables are filled to size with the bulk paths (kgi_fill_sorted, kgx_dpt_load) with distinct random entries, then timed
inserts of fresh records (all ADD_OK, the common case) alternate between the two tables, batch for batch."""
import argparse
import json
import os
import re
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from kangaroo_b200.dptable import DeviceDPTable, HASH_SIZE, memory_bytes  # noqa: E402
from kangaroo_b200.ingest import DPTable  # noqa: E402

DP40 = np.dtype([("kidx", "<u4"), ("h", "<u4"), ("x", "<u8", 2), ("d", "<u8", 2)])
KEY = (0x79BE667EF9DCBBAC55A06295CE870B07029BFCDB2DCE28D959F2815B16F81798,
       0x483ADA7726A3C4655DA4FBFC0E1108A8FD17B448A68554199C47D08FFB10D4B8)


def emit(**kw):
    print(json.dumps(kw), flush=True)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,memory.total", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q


def fill(size, dev, host, rng, per_chunk=4096):
    """size distinct entries in work-file order, bucket by bucket, into both tables"""
    m = size // HASH_SIZE
    extra = size - m * HASH_SIZE
    for b0 in range(0, HASH_SIZE, per_chunk):
        nb = min(per_chunk, HASH_SIZE - b0)
        counts = np.full(nb, m, dtype=np.int64)
        if b0 < extra:
            counts[:min(nb, extra - b0)] += 1
        n = int(counts.sum())
        if n == 0:
            continue
        h = np.repeat(np.arange(b0, b0 + nb, dtype=np.uint32), counts)
        x1 = rng.integers(0, 1 << 63, n, dtype=np.uint64) * np.uint64(2)       # even: fresh inserts use odd x[1]
        order = np.lexsort((x1, h))
        e = np.empty((n, 4), dtype=np.uint64)
        e[:, 1] = x1[order]
        e[:, 0] = rng.integers(0, 1 << 63, n, dtype=np.uint64)
        e[:, 2:] = rng.integers(0, 1 << 62, (n, 2), dtype=np.uint64)
        host.fill_sorted(h, e)
        dev.load(h, e)


def fresh(rng, n):
    r = np.zeros(n, dtype=DP40)
    r["h"] = rng.integers(0, HASH_SIZE, n)
    r["x"] = rng.integers(0, 1 << 63, (n, 2), dtype=np.uint64)
    r["x"][:, 1] = r["x"][:, 1] * np.uint64(2) + np.uint64(1)
    r["d"] = rng.integers(0, 1 << 62, (n, 2), dtype=np.uint64)
    return r


def bench_size(torch, size, batches, reps, rng, tmp):
    cap = max(int(size * 1.3) + 16 * max(batches) * reps, 1 << 20)
    dev, host = DeviceDPTable(0, cap), DPTable(threads=0)
    t0 = time.perf_counter()
    fill(size, dev, host, rng)
    emit(what="fill", entries=size, seconds=round(time.perf_counter() - t0, 2), device_capacity=cap,
         device_bytes=memory_bytes(cap), bytes_per_entry_of_capacity=round(memory_bytes(cap) / cap, 2))
    stream = torch.cuda.current_stream()
    for nb in batches:
        td, th = [], []
        for _ in range(reps):                                       # alternated, batch for batch
            recs = fresh(rng, nb)
            buf = torch.from_numpy(recs.view(np.uint8)).cuda()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            dev.insert(buf.data_ptr(), [nb], 0, stream.cuda_stream)
            dev.events()
            td.append(time.perf_counter() - t0)
            t0 = time.perf_counter()
            host.add_dp40(recs.view(np.uint8))
            th.append(time.perf_counter() - t0)
        emit(what="insert", entries=size, batch=nb, reps=reps, device_rec_per_s=round(nb / np.median(td)),
             host_rec_per_s=round(nb / np.median(th)), host_threads=host.threads,
             device_ms=round(1e3 * np.median(td), 3), host_ms=round(1e3 * np.median(th), 3))
    n = len(host)
    assert dev.count() == n
    # checkpoint table part: host writes its table; the device exports in work-file order, kgi_fill_sorted, the same writer
    path = os.path.join(tmp, "t.work")
    t0 = time.perf_counter()
    host.save_work(path, 12, 1, 2, KEY)
    t_host = time.perf_counter() - t0
    host.reset()
    t0 = time.perf_counter()
    dev.export_begin(stream.cuda_stream)
    k = sum(e.shape[0] for _h, e in dev.export_chunks())
    dev.export_end()
    t_exp = time.perf_counter() - t0
    assert k == n
    t0 = time.perf_counter()
    dev.to_host(host, stream.cuda_stream)
    t_fill = time.perf_counter() - t0
    t0 = time.perf_counter()
    host.save_work(path, 12, 1, 2, KEY)
    t_write = time.perf_counter() - t0
    os.unlink(path)
    emit(what="export", entries=n, device_export_s=round(t_exp, 3), device_export_fill_s=round(t_fill, 3),
         write_s=round(t_write, 3), host_table_write_s=round(t_host, 3))
    dev.close(); host.close()


def solver_runs(gpus, dps, max_steps, rounds, cfg):
    res = {}
    for rnd in range(rounds):
        for dp in dps:
            for kind in ("host", "device"):
                env = dict(os.environ, KGX_DPTABLE=kind)
                cmd = ([sys.executable, "-m", "torch.distributed.run", "--standalone", "--nproc-per-node", str(gpus)] if gpus > 1
                       else [sys.executable]) + ["-m", "kangaroo_b200.solver", cfg, "--dp", str(dp), "--seed", str(100 + rnd),
                                                 "--max-steps", str(max_steps)]
                out = subprocess.run(cmd, capture_output=True, text=True, cwd=ROOT, env=env, timeout=3600)
                txt = out.stdout + out.stderr
                m = re.search(r"Solver rate: (\d+) MJump/s steady state.*?over all (\d+) steps \(([\d.]+) s\); rank-0 ingest ([\d.]+) ms/step; (\d+) DPs", txt)
                if not m:
                    emit(what="solver", gpus=gpus, dp=dp, table=kind, error=txt[-1500:])
                    continue
                rate, steps, secs, ingest, ndp = int(m.group(1)), int(m.group(2)), float(m.group(3)), float(m.group(4)), int(m.group(5))
                res.setdefault((dp, kind), []).append(rate)
                emit(what="solver", gpus=gpus, dp=dp, table=kind, round=rnd, steady_mjump_s=rate, steps=steps,
                     ms_per_step=round(1e3 * secs / steps, 2), rank0_table_ms_per_step=ingest, dps=ndp,
                     lost="items lost" in txt, table_line=(re.search(r"DP table: .*", txt) or [""])[0])
    for (dp, kind), v in sorted(res.items()):
        emit(what="solver_summary", gpus=gpus, dp=dp, table=kind, median_mjump_s=float(np.median(v)), runs=len(v))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="1e7,1e8,6e8")
    ap.add_argument("--batches", default="38000,606000")
    ap.add_argument("--reps", type=int, default=8)
    ap.add_argument("--solver", action="store_true")
    ap.add_argument("--gpus", type=int, default=0, help="solver ranks (0 = every visible GPU)")
    ap.add_argument("--dps", default="16,12")
    ap.add_argument("--max-steps", type=int, default=600)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--config", default=os.path.join(ROOT, "tests", "golden", "puzzle110_window80.txt"))
    a = ap.parse_args()
    import torch
    emit(what="card", gpus=card())
    rng = np.random.default_rng(1)
    with tempfile.TemporaryDirectory() as tmp:
        for s in [int(float(v)) for v in a.sizes.split(",") if float(v) > 0]:
            bench_size(torch, s, [int(v) for v in a.batches.split(",")], a.reps, rng, tmp)
    if a.solver:
        solver_runs(a.gpus or torch.cuda.device_count(), [int(v) for v in a.dps.split(",")], a.max_steps, a.rounds, a.config)


if __name__ == "__main__":
    main()
