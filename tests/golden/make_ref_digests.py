"""Record tests/golden/ref_digests.json: the digest of the reference's own outputs (oracle/_ref/libkref.so, i.e. the reference's
SECPK1 sources driven by oracle/ref_harness.cpp) for every case of tests/test_oracle_vs_ref.py.  Run from the repository root
where the reference build exists:  python tests/golden/make_ref_digests.py"""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from oracle import kgo  # noqa: E402
from tests import test_oracle_vs_ref as t  # noqa: E402


def main():
    ref = kgo.Reference()
    out = {name: t.digest(run(ref, True)) for name, run in sorted(t.RUNS.items())}
    with open(t.GOLDEN, "w") as f:
        json.dump(out, f, indent=1, sort_keys=True)
        f.write("\n")


if __name__ == "__main__":
    main()
