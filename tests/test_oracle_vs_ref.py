"""Pin oracle/kgx_oracle.c against the reference's own SECPK1 code (oracle/_ref/libkref.so, built from the reference sources
by oracle/Makefile).  Each case runs the same calls on the oracle and on the reference.  Where the reference build is absent
the oracle's outputs are checked against the digest of the reference's outputs for the same calls, recorded in
tests/golden/ref_digests.json by tests/golden/make_ref_digests.py."""
import hashlib
import json
import os
import random

import numpy as np
import pytest

from oracle import kgo

P, N = kgo.P, kgo.N
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_digests.json")
KEY64 = 0x5B3F38AF935A3640D158E871CE6E9666DB862636383386EE510F18CCC3BD72EB


def _canon(v):
    if isinstance(v, np.ndarray):
        return _canon(v.tolist())
    if isinstance(v, (list, tuple)):
        return [_canon(x) for x in v]
    if isinstance(v, (int, np.integer)):
        return "%x" % int(v)
    return v


def digest(v):
    return hashlib.sha256(json.dumps(_canon(v)).encode()).hexdigest()


@pytest.fixture(scope="session")
def live_reference():
    return kgo.Reference() if kgo.reference_available() else None


def agrees(name, oracle, reference):
    """The outputs of RUNS[name] on the oracle equal the reference's: live where the reference build exists, and always
    against the recorded digest of the reference's outputs."""
    got = RUNS[name](oracle, False)
    if reference is not None:
        assert _canon(got) == _canon(RUNS[name](reference, True))
    assert digest(got) == json.load(open(GOLDEN))[name]
    return got


def _field_ops(be, ref):
    rng = random.Random(3)
    edge = [0, 1, 2, P - 1, P - 2, 0x1000003D1, 2**255, 2**256 - 1 - 0x1000003D1, 2**128 - 1]
    vals = edge + [rng.randrange(P) for _ in range(3000)]
    out = [(be.mod_mul(a, b), be.mod_sqr(a), be.mod_sub(a, b)) for a, b in zip(vals[:-1], vals[1:])]
    return out + [be.mod_inv(a) for a in vals[:300]]


def _order_ops(be, ref):
    rng = random.Random(4)
    out = []
    for _ in range(500):
        a, b = rng.randrange(N), rng.randrange(N)
        out.append((be.order_add(a, b), be.order_sub(a, b)))
    return out


def _rng_and_rand(be, ref):
    out = []
    for seed in (0, 1, 0x600DCAFE, 0xFFFFFFFF):
        be.rseed(seed)
        out.append([be.rndl() for _ in range(700)])
        out.append([be.rand_bits(nbit) for nbit in (1, 31, 32, 33, 64, 65, 128, 255, 256)])
    return out


def _scalar_mult_and_add(be, ref):
    rng = random.Random(5)
    ks = [1, 2, 3, 255, 256, 257, 2**64, N - 1, N - 2] + [rng.randrange(1, N) for _ in range(40)]
    pts = [be.ec_mul_g(k) for k in ks]
    return pts + [be.ec_add(a, b) for a, b in zip(pts[:-1], pts[1:]) if a[0] != b[0]]


def _jump_tables(be, ref):
    out = []
    for rp in (32, 40, 48, 56, 64, 72, 80, 84, 110, 115, 125, 256):
        out.append((rp, be.create_jump_table(rp), be.last_draws))
    return out


def _herd_and_jump_loop(be, ref):
    table = kgo.Oracle().create_jump_table(64)
    key = kgo.Oracle().ec_mul_g(KEY64)
    out = []
    for first_type in (0, 1):
        be.rseed(42)
        herd = be.create_herd(300, 64, 2**63 - 1, key, first_type)
        out.append([v.copy() for v in herd])
    dps = be.jump_cpu(*herd, table, 70, kgo.Oracle().dp_mask(6), grp=1024 if ref else 128)
    out += [herd, sorted(dps)]
    # Check.cpp single-AddDirect replay
    be.rseed(42)
    x, y, d = (kgo.from_limbs(v[7]) for v in be.create_herd(8, 64, 2**63 - 1, key, 0))
    for _ in range(20):
        x, y, d = be.jump_single(x, y, d, table)
    return out + [(x, y, d)]


def _hash_convert(be, ref):
    rng = random.Random(6)
    out = []
    for _ in range(200):
        x = rng.randrange(P)
        d = rng.randrange(2**126) if rng.random() < 0.5 else N - rng.randrange(1, 2**126)
        out.append(be.hash_convert(x, d, rng.randrange(2)))
    return out


def _symmetric_jump_table(rp):
    def run(be, ref):
        return be.create_jump_table_sym(rp), be.last_uv, be.last_draws
    return run


def _symmetric_herd_and_walk(be, ref):
    rp = 64
    key = kgo.Oracle().ec_mul_g(0x5B3F38AF935A3640D158E871CE6E9666DB862636383386EE0000000000123000)
    wdiv4 = ((1 << rp) - 1) >> 2
    table = kgo.Oracle().create_jump_table_sym(rp)
    n = 96
    be.rseed(777)
    x, y, d = be.create_herd_sym(n, rp, wdiv4, key, 0)
    out = [(x.copy(), y.copy(), d.copy())]
    mask = kgo.Oracle().dp_mask(4)
    for rule, init in (("lastjump", 32), ("symclass", 0)):
        state = np.full(n, init, dtype=np.uint8)
        dps = be.jump_sym(x, y, d, state, table, 200, mask, grp=24 if ref else 32, rule=rule)
        out.append((x.copy(), y.copy(), d.copy(), state.copy(), sorted(dps)))
    return out


SYM_RANGE_POWERS = [40, 56, 64, 80, 109, 125]
RUNS = {"field_ops": _field_ops, "order_ops": _order_ops, "rng_and_rand": _rng_and_rand,
        "scalar_mult_and_add": _scalar_mult_and_add, "jump_tables": _jump_tables, "herd_and_jump_loop": _herd_and_jump_loop,
        "hash_convert": _hash_convert, "symmetric_herd_and_walk": _symmetric_herd_and_walk}
RUNS.update({"symmetric_jump_table_%d" % rp: _symmetric_jump_table(rp) for rp in SYM_RANGE_POWERS})


def test_field_ops(oracle, live_reference):
    agrees("field_ops", oracle, live_reference)


def test_order_ops(oracle, live_reference):
    agrees("order_ops", oracle, live_reference)


def test_rng_and_rand(oracle, live_reference):
    agrees("rng_and_rand", oracle, live_reference)


def test_scalar_mult_and_add(oracle, live_reference):
    agrees("scalar_mult_and_add", oracle, live_reference)


def test_jump_tables_all_range_powers(oracle, live_reference):
    agrees("jump_tables", oracle, live_reference)


def test_herd_and_jump_loop(oracle, live_reference):
    out = agrees("herd_and_jump_loop", oracle, live_reference)
    assert len(out[3]) > 200


def test_hash_convert(oracle, live_reference):
    agrees("hash_convert", oracle, live_reference)


# ---- USE_SYMMETRY restatement (SURVEY 8f/f4) pinned to the reference's own Int / Secp256K1 code -------------------------
@pytest.mark.parametrize("rp", SYM_RANGE_POWERS)
def test_symmetric_jump_table_matches_reference(oracle, live_reference, rp):
    """Kangaroo.cpp:742-832 USE_SYMMETRY branch: the two primes u, v come from Int::IsProbablePrime, whose Miller-Rabin bases
    are drawn from the same MT19937 stream as the distances -- the oracle reproduces that consumption exactly."""
    (jd, _, _), (u, v), _ = agrees("symmetric_jump_table_%d" % rp, oracle, live_reference)
    assert all(int(jd[i, 0]) % u == 0 for i in range(16)) and all(int(jd[i, 0]) % v == 0 for i in range(16, 32))


def test_symmetric_herd_and_walk_match_reference(oracle, live_reference):
    """CreateHerd (Kangaroo.cpp:670-738, sym branch) and the symmetric walk Check.cpp:534-556 replays (lastJump limiter,
    ModPositiveK1 class switch, d = n - d): oracle (batched inverse) == reference (one AddDirect per jump), bit for bit."""
    out = agrees("symmetric_herd_and_walk", oracle, live_reference)
    key = oracle.ec_mul_g(0x5B3F38AF935A3640D158E871CE6E9666DB862636383386EE0000000000123000)
    n = 96
    oy, od = out[0][1], out[0][2]
    half = (kgo.P - 1) // 2
    assert all(kgo.from_limbs(oy[i]) <= half for i in range(n))
    assert any(kgo.from_limbs(od[i]) > kgo.N // 2 for i in range(n))           # some distances went negative (mod n)
    for rule, (ox, _, od, lo, dps) in zip(("lastjump", "symclass"), out[1:]):
        assert len(dps) > 500, rule
        if rule == "symclass":
            assert set(np.unique(lo)) == {0, 1}
    # invariant of the class walk: tame x == (d*G).x ; wild x == (key + d*G).x or (key - d*G).x -- a class switch negates
    # the whole point, i.e. d AND the key term, which is why CheckKey tries +-key and the four sign pairs (Kangaroo.cpp:218-253)
    for i in (0, 1, 2, 3, 50, 95):
        dv = kgo.from_limbs(od[i])
        if i % 2 == 0:
            assert oracle.ec_mul_g(dv)[0] == kgo.from_limbs(ox[i])
        else:
            cands = (oracle.ec_add(key, oracle.ec_mul_g(dv))[0], oracle.ec_add(key, oracle.ec_mul_g(N - dv))[0])
            assert kgo.from_limbs(ox[i]) in cands
