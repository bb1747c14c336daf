"""Cost of the solver's checkpoints on the default grid (296 x 128 x 128 = 4.85 M kangaroos per GPU, in80, dp 16):

  1. walk export: kgx_walks_begin + kgx_walks_read of the whole herd into pinned memory (device conversion + D2H), GB/s
  2. import + verification of the same records (kgx_walks_load, one scalar multiplication per walk)
  3. the solver with --work-interval S --save-kangaroos against the same run without checkpoints, alternated; the
     checkpoint lines give wall time and step-loop stall, the summary lines the steady rate
     (with --gpus N > 1 the solver runs under torchrun on N GPUs)

  python scripts/bench_checkpoint.py --out profiles/r3_checkpoint.txt [--steps 3400 --interval 60 --rounds 2 --gpus 1]
"""
import argparse
import os
import re
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip() or "nvidia-smi unavailable"


def walks_io(log):
    import torch
    from kangaroo_b200 import GPUEngine, random_herd_arrays
    from kangaroo_b200 import ecmath as ec
    eng = GPUEngine(296, 128, 0, 1 << 17)
    n = eng.nbKangaroo
    key = ec.mul(0x1234567)
    eng.SetWildOffset(1 << 79)
    sc, d128 = random_herd_arrays(n, 80, 1 << 79, np.random.Generator(np.random.PCG64(5)))
    eng.CreateHerdRaw(sc, d128, key)
    host = torch.empty(n * 96, dtype=torch.uint8).pin_memory()
    times = []
    for _ in range(4):
        t0 = time.perf_counter()
        eng.WalksBegin()
        eng.WalksRead(host)
        times.append(time.perf_counter() - t0)
        eng.WalksEnd()
    t = min(times[1:])
    log("walk export, %d walks (%.1f MB): %.1f ms = %.2f GB/s (device conversion + D2H into pinned memory; best of 3 after a warm-up)"
        % (n, n * 96 / 1e6, t * 1e3, n * 96 / t / 1e9))
    recs = host.numpy()
    vt = []
    for _ in range(2):
        t0 = time.perf_counter()
        nb, _ = eng.LoadWalks(recs, key=key)
        vt.append(time.perf_counter() - t0)
        assert nb == 0
    t0 = time.perf_counter()
    eng.LoadWalks(recs, verify=False)
    ti = time.perf_counter() - t0
    log("walk import alone: %.1f ms; import + verification: %.1f ms (%.1f M walks/s checked)" % (ti * 1e3, min(vt) * 1e3, n / min(vt) / 1e6))
    eng.close()


def solver_run(args, gpus, work):
    cmd = [sys.executable, "-m", "kangaroo_b200.solver"] if gpus == 1 else \
        [sys.executable, "-m", "torch.distributed.run", "--standalone", "--nproc-per-node", str(gpus), "-m", "kangaroo_b200.solver"]
    cmd += [os.path.join(ROOT, "tests", "golden", "in80.txt"), "--dp", "16", "--seed", "1"] + args
    if work:
        cmd += ["--work-file", work]
    p = subprocess.run(cmd, capture_output=True, text=True, cwd=ROOT)
    return p.stdout + p.stderr


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="")
    ap.add_argument("--steps", type=int, default=3400)
    ap.add_argument("--interval", type=float, default=60)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--skip-io", action="store_true")
    a = ap.parse_args()
    lines = []

    def log(s):
        print(s, flush=True)
        lines.append(s)
    log("card: %s" % card())
    if not a.skip_io:
        walks_io(log)
    with tempfile.TemporaryDirectory() as tmp:
        work = os.path.join(tmp, "bench.work")
        rates = {"off": [], "on": []}
        for r in range(a.rounds):
            for mode in ("off", "on"):
                extra = ["--max-steps", str(a.steps)]
                if mode == "on":
                    extra += ["--work-interval", str(a.interval), "--save-kangaroos"]
                out = solver_run(extra, a.gpus, work if mode == "on" else "")
                m = re.search(r"Solver rate: (\d+) MJump/s steady state", out)
                ck = re.findall(r"checkpoint: .*", out)
                rates[mode].append(int(m.group(1)) if m else 0)
                log("round %d, checkpoints %s, %d GPU(s): %s MJump/s steady; %s" %
                    (r, mode, a.gpus, m.group(1) if m else "?", "key found" if "Priv:" in out else "no key"))
                for c in ck:
                    log("    " + c)
                if not m:
                    log(out[-1500:])
            if os.path.exists(work):
                os.unlink(work)
        off, on = np.mean(rates["off"]), np.mean(rates["on"])
        log("mean steady rate: %.0f MJump/s without, %.0f MJump/s with checkpoints every %.0f s: %+.2f %%"
            % (off, on, a.interval, 100.0 * (on - off) / max(off, 1)))
    if a.out:
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
