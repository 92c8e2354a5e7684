"""GPU parity of the building blocks through the C ABI: PTX field arithmetic, hash_to_G2, aggregateAll."""
import ctypes as C
import hashlib
import json
import os
import random

import pytest

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden")
P = 0x1a0111ea397fe69a4b1ba7b6434bacd764774b84f38512bf6730d2a0f6b0f6241eabfffeb153ffffb9feffffffffaaab


def _fp_inv_mont(x48):
    """blst_fp_inverse on a Montgomery-form input: the Montgomery form of the inverse, R^2 / x mod p (0 -> 0)."""
    x = int.from_bytes(x48, "little")
    return (pow(x, -1, P) * (1 << 768) % P if x else 0).to_bytes(48, "little")


def test_fp_ptx_vs_blst(cache):
    import nim_blscurve_b200 as bg
    rng = random.Random(99)
    n = 2048
    edge = [0, 1, P - 1, P - 2, 2 ** 380, (P - 1) // 2, 2 ** 32 - 1, 2 ** 383 % P]
    a = [edge[i % len(edge)] if i < 64 else rng.randrange(P) for i in range(n)]
    b = [edge[(i // 8) % len(edge)] if i < 64 else rng.randrange(P) for i in range(n)]
    ab = b"".join(x.to_bytes(48, "little") for x in a)
    bb = b"".join(x.to_bytes(48, "little") for x in b)
    R = 1 << 384
    Rinv = pow(R, -1, P)
    for op, name, fn in ((0, "mul", lambda x, y: x * y * Rinv % P), (1, "add", lambda x, y: (x + y) % P),
                         (2, "sub", lambda x, y: (x - y) % P), (3, "sqr", lambda x, y: x * x * Rinv % P)):
        out = (C.c_uint8 * (48 * n))()
        assert bg.lib().blsgpu_test_fp(cache.handle, op, ab, bb, n, out) == 0
        got = bytes(out)
        for i in range(n):
            assert int.from_bytes(got[48 * i:48 * i + 48], "little") == fn(a[i], b[i]), (name, i)
        # and bit-exact (canonical 48-byte encoding) on a sample
        for i in range(0, n, 97):
            assert got[48 * i:48 * i + 48] == fn(a[i], b[i]).to_bytes(48, "little")
    # the binary-Euclid inversion of the single-thread tails
    out = (C.c_uint8 * (48 * n))()
    assert bg.lib().blsgpu_test_fp(cache.handle, 6, ab, None, n, out) == 0
    got = bytes(out)
    for i in range(0, n, 13):
        assert got[48 * i:48 * i + 48] == _fp_inv_mont(ab[48 * i:48 * i + 48]), ("inv_vartime", i)
    out = (C.c_uint8 * (48 * 64))()
    assert bg.lib().blsgpu_test_fp(cache.handle, 4, ab[48 * 64:48 * 128], None, 64, out) == 0
    for i in range(64):
        assert bytes(out)[48 * i:48 * i + 48] == _fp_inv_mont(ab[48 * (64 + i):48 * (65 + i)])


def test_hash_to_g2_eth2_dst(cache, br):
    import nim_blscurve_b200 as bg
    dst = b"BLS_SIG_BLS12381G2_XMD:SHA-256_SSWU_RO_POP_"
    msgs = b"".join(hashlib.sha256(b"m%d" % i).digest() for i in range(300))
    comp, aff = bg.hashToG2(cache, msgs, 32, dst)
    rcomp, raff = br.hash_to_g2(msgs, 32, dst)
    assert comp == rcomp and aff == raff


def test_hash_to_g2_rfc9380_vectors(cache):
    """Golden vectors of the reference: vendor/blst/bindings/vectors/hash_to_curve/BLS12381G2_XMD_SHA-256_SSWU_RO_.json"""
    import nim_blscurve_b200 as bg
    from oracle import pyref as pr
    d = json.load(open(os.path.join(GOLD, "BLS12381G2_XMD_SHA-256_SSWU_RO_.json")))
    dst = d["dst"].encode()
    for v in d["vectors"]:
        m = v["msg"].encode()
        comp, aff = bg.hashToG2(cache, m, len(m), dst)
        x = tuple(int(t, 16) for t in v["P"]["x"].split(","))
        y = tuple(int(t, 16) for t in v["P"]["y"].split(","))
        assert pr.g2_from_mem(aff) == (x, y)
        assert comp == pr.g2_compress((x, y))


@pytest.mark.parametrize("n", [1, 2, 3, 128, 512])
def test_aggregate_all(cache, br, n):
    import nim_blscurve_b200 as bg
    sets = br.make_sets(500, min(n, 24))
    pks = [sets[i:i + 96] for i in range(0, len(sets), 320)]
    sigs = [sets[i + 128:i + 320] for i in range(0, len(sets), 320)]
    pks = (pks * (n // len(pks) + 1))[:n]           # repeats exercise the doubling path
    sigs = (sigs * (n // len(sigs) + 1))[:n]
    assert bg.aggregateAll(cache, pks) == br.aggregate_g1(b"".join(pks))
    assert bg.aggregateAll(cache, sigs) == br.aggregate_g2(b"".join(sigs))
    assert bg.aggregateAll(cache, []) == (False, b"")


@pytest.mark.parametrize("n", [1, 2, 5, 127, 512])
def test_subtract_all(cache, br, n):
    """subtractAll (blst_min_pubkey_sig_core.nim:197-209) against BLST's from_affine / add_or_double_affine / cneg chain."""
    import nim_blscurve_b200 as bg
    sets = br.make_sets(700, 24)
    pks = [sets[i:i + 96] for i in range(0, len(sets), 320)]
    sigs = [sets[i + 128:i + 320] for i in range(0, len(sets), 320)]
    _, dpk = br.aggregate_g1(b"".join(pks))
    _, dsig = br.aggregate_g2(b"".join(sigs))
    epk, esig = (pks * (n // len(pks) + 1))[:n], (sigs * (n // len(sigs) + 1))[:n]
    assert bg.subtractAll(cache, dpk, epk) == br.subtract_all(dpk, b"".join(epk))
    assert bg.subtractAll(cache, dsig, esig) == br.subtract_all(dsig, b"".join(esig))
    # dst at infinity, and an empty list (dst untouched, :199-200)
    assert bg.subtractAll(cache, bytes(96), epk) == br.subtract_all(bytes(96), b"".join(epk))
    assert bg.subtractAll(cache, dsig, []) == dsig


def test_subtract_all_golden_and_infinity(cache):
    import json, os
    import nim_blscurve_b200 as bg
    a = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "aggregate.json")))
    pk, sg = bytes.fromhex(a["pubkeys"]), bytes.fromhex(a["signatures"])
    pks, sgs = [pk[i:i + 96] for i in range(0, len(pk), 96)], [sg[i:i + 192] for i in range(0, len(sg), 192)]
    assert bg.subtractAll(cache, bytes.fromhex(a["agg_pubkey"]), pks[:5]).hex() == a["sub5_pubkey"]
    assert bg.subtractAll(cache, bytes.fromhex(a["agg_signature"]), sgs[:5]).hex() == a["sub5_signature"]
    assert bg.subtractAll(cache, bytes.fromhex(a["agg_pubkey"]), pks) == bytes(96)          # P - P = infinity
    assert bg.subtractAll(cache, sgs[0], sgs[:1]) == bytes(192)


def test_imad_peak_runs(cache):
    import nim_blscurve_b200 as bg
    r = bg.lib().blsgpu_imad_peak(cache.handle, 1)
    assert r > 1e11


def test_small_route_hash_matches_blst(cache, br):
    """The message hash of the small-batch route (two-lane SSWU kernel + cofactor clearing as a per-set dataflow program
    over complete projective formulas) against BLST's hash_to_g2 on 300 messages."""
    import ctypes as C
    import nim_blscurve_b200 as bg
    from oracle import pyref as pr
    n = 300
    sets = br.make_sets(5, n)
    hout = (C.c_uint8 * (n * 288))()
    assert bg.lib().blsgpu_test_small_hash(cache.handle, sets, n, None, hout) == 0
    msgs = b"".join(sets[i * 320 + 96:i * 320 + 128] for i in range(n))
    ref = br.hash_to_g2(msgs, 32, pr.DST_ETH2)[1]
    raw = bytes(hout)
    for i in range(n):
        v = [pr.fp_from_mont_bytes(raw[i * 288 + 48 * k:i * 288 + 48 * k + 48]) for k in range(6)]
        zi = pr.f2_inv((v[4], v[5]))
        got = (pr.f2_mul((v[0], v[1]), zi), pr.f2_mul((v[2], v[3]), zi))
        assert pr.g2_to_mem(got) == ref[i * 192:(i + 1) * 192], i
