"""-m gpu: the reference's UNMODIFIED host program (main/Kangaroo/Check/HashTable/SECPK1, compiled from
the reference sources by oracle/build_dropin.sh) linked against the B200 engine through the GPUEngine shim.
  * `-check`  = the reference's own parity test, Check.cpp:467-621 (GPU vs CPU after NB_RUN jumps + DP set)
  * in56 / in64 = end-to-end solves with published answers (README.md:146-147, 194-195)
The binary is built in the build container (the reference sources do not exist on the GPU box) and travels."""
import os
import subprocess

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "oracle", "_ref", "kangaroo_b200")
GOLD = os.path.join(ROOT, "tests", "golden")


def run(args, timeout=600, env=None):
    if not os.path.exists(BIN):
        pytest.skip("oracle/_ref/kangaroo_b200 not built (needs the reference sources at build time)")
    e = dict(os.environ)
    e.update(env or {})
    p = subprocess.run([BIN] + args, capture_output=True, text=True, timeout=timeout, cwd=ROOT, env=e)
    return p.stdout + p.stderr


def test_reference_check_gpu_vs_cpu():
    out = run(["-gpu", "-check", "-g", "8,128"])       # 131072 kangaroos -> ~32k DPs at dp=8 (< 65536 buffer)
    assert "CPU/GPU ok" in out, out[-3000:]
    assert "DP Mismatch" not in out and "not ok" not in out


@pytest.mark.parametrize("env", [{"KGX_MODE": "stream", "KGX_STREAM_G": "128"}, {"KGX_MODE": "resident"}, {"KGX_MODE": "tmem"}],
                         ids=["stream128", "resident", "tmem"])
def test_reference_check_largest_grid_on_each_kernel(env):
    """Check.cpp hard-codes dp = 8 and a 65536-record DP buffer (:417, :492), so the largest herd its DP comparison can
    hold is ~2.6e5 kangaroos (expected DPs = nb * 64 / 256 < 65536): `-g 15,128` = 245,760 kangaroos -> ~61.4 k DPs.
    Run on the benchmarked stream kernel (G = 128, as on the default grid), the adaptive group size, and the tile kernel."""
    out = run(["-gpu", "-check", "-g", "15,128"], timeout=1200, env=env)
    assert "CPU/GPU ok" in out, out[-3000:]
    assert "DP Mismatch" not in out and "not ok" not in out and "items lost" not in out


def test_reference_check_odd_grid():
    out = run(["-gpu", "-check", "-g", "3,32"])
    assert "CPU/GPU ok" in out, out[-3000:]


def test_solve_in56():
    out = run(["-t", "0", "-gpu", "-g", "16,128", os.path.join(GOLD, "in56.txt")])
    assert "CD612C0F05F3DA03" in out.upper().replace(" ", ""), out[-2000:]


def test_solve_in64():
    out = run(["-t", "0", "-gpu", "-g", "64,128", os.path.join(GOLD, "in64.txt")], timeout=900)
    assert "5B3F38AF935A3640D158E871CE6E9666DB862636383386EE510F18CCC3BD72EB" in out.upper(), out[-2000:]


def test_checkpoint_round_trip_through_reference_work_files(tmp_path):
    """SURVEY 8f/f3: `-w f -wi N -ws` makes the reference's Thread.cpp:330-335 request a save, SolveKeyGPU calls
    GPUEngine::GetKangaroos (Kangaroo.cpp:618-626) and Backup.cpp:449-572 writes HEADW + hash table + every kangaroo; `-i f`
    reads it back (Backup.cpp:291-364) and the search goes on from the saved herd through SetKangaroos.  Everything but the
    engine is the reference's own code, so passing means the engine's Get/SetKangaroos round trip is exact at full size
    (4.85 M kangaroos, 466 MB of walks).  Run 1 saves at every status tick (`-wi 1`: Timer::get_tick() counts from program
    start, Thread.cpp:330-335) and gives up at 25 % of the expected operations (-m); `-wcheck` validates every stored DP (d*G [+P] == x); run 2 resumes from the file and must find the key."""
    work = str(tmp_path / "k.work")
    cfg = os.path.join(GOLD, "puzzle110_window72.txt")
    out1 = ""
    for attempt in range(3):                                          # a lucky run may solve before the first save
        out1 = run(["-t", "0", "-gpu", "-d", "14", "-w", work, "-wi", "1", "-ws", "-m", "0.25", cfg], timeout=600)
        if os.path.exists(work) and "Aborted" in out1:
            break
    assert os.path.exists(work) and "SaveWork" in out1 and "Aborted" in out1, out1[-2000:]
    assert os.path.getsize(work) > 4849664 * 96                       # the whole default herd is in the file
    chk = run(["-wcheck", work], timeout=600)
    assert "[100.000% OK]" in chk and "Wrong" not in chk, chk[-1500:]         # Check.cpp:393-409
    out2 = run(["-t", "0", "-gpu", "-i", work], timeout=900)
    assert "FectchKangaroos" in out2 and "kangaroos loaded" in out2, out2[-2000:]
    assert "35C0D7234DF7DEB0F20CF7062444" in out2.upper(), out2[-2000:]
