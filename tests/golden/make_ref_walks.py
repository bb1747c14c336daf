"""Record tests/golden/ref_walks_in80.work.gz: a work file with kangaroos (-ws) written by the reference's CPU program
(oracle/_ref/kangaroo_ref_cpu, built by oracle/Makefile) on the in80 range -- 2 threads x 1024 kangaroos, DP 20 so that the
table stays nearly empty, stopped by -m after its first periodic save.  tests/test_checkpoint_cpu.py reads it to pin the
walk-record format and the distance convention (wild distances below zero stored as n - |d|).  Run from the repository
root where the reference build exists:  python tests/golden/make_ref_walks.py"""
import gzip
import os
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
REFBIN = os.path.join(ROOT, "oracle", "_ref", "kangaroo_ref_cpu")
OUT = os.path.join(ROOT, "tests", "golden", "ref_walks_in80.work.gz")


def main():
    if not os.path.exists(REFBIN):
        sys.exit("%s is missing: build it with make -C oracle ref" % REFBIN)
    with tempfile.TemporaryDirectory() as tmp:
        work = os.path.join(tmp, "ref.work")
        subprocess.run([REFBIN, "-t", "2", "-d", "20", "-w", work, "-ws", "-wi", "1", "-m", "0.000003",
                        os.path.join(ROOT, "tests", "golden", "in80.txt")], check=True, timeout=300, cwd=tmp)
        with open(work, "rb") as f, gzip.GzipFile(OUT, "wb", compresslevel=9, mtime=0) as g:
            g.write(f.read())
    print("wrote", OUT)


if __name__ == "__main__":
    main()
