"""CPU: the device arithmetic headers (nim_blscurve_b200/csrc/*.cuh) compiled as plain C++ (tests/hostsim) and
checked against the golden fixtures.  This exercises every formula the kernels use (tower, curves, SSWU/isogeny/
cofactor, Miller loop, final exponentiation, the whole batch pipeline order) except the PTX bodies of fp.cuh,
which the GPU tests cover."""
import ctypes as C
import json
import os
import random
import subprocess

import pytest

from oracle import pyref as pr

HERE = os.path.dirname(os.path.abspath(__file__))
GOLD = os.path.join(HERE, "golden")
SO = os.path.join(HERE, "hostsim", "libhostsim.so")
P = pr.P


@pytest.fixture(scope="module")
def hs():
    src = os.path.join(HERE, "hostsim", "hostsim.cpp")
    csrc = os.path.join(os.path.dirname(HERE), "nim_blscurve_b200", "csrc")
    deps = [src] + [os.path.join(csrc, f) for f in os.listdir(csrc) if f.endswith((".cuh", ".hpp"))]
    if not os.path.exists(SO) or any(os.path.getmtime(d) > os.path.getmtime(SO) for d in deps):
        subprocess.run(["g++", "-O2", "-shared", "-fPIC", "-x", "c++", "-std=c++17", "-o", SO, src], check=True)
    return C.CDLL(SO)


def buf(b):
    return (C.c_uint8 * len(b)).from_buffer_copy(b)


def out(n):
    return (C.c_uint8 * n)()


def test_fp_ops(hs):
    rng = random.Random(1)
    Rinv = pow(1 << 384, -1, P)
    for it in range(500):
        a, b = rng.randrange(P), rng.randrange(P)
        if it < 4:
            a, b = [(0, 0), (1, P - 1), (P - 1, P - 1), (P - 1, 1)][it]
        r = out(48)
        ab, bb = buf(a.to_bytes(48, "little")), buf(b.to_bytes(48, "little"))
        hs.hs_fp_mul(ab, bb, r)
        assert int.from_bytes(bytes(r), "little") == a * b * Rinv % P
        hs.hs_fp_add(ab, bb, r)
        assert int.from_bytes(bytes(r), "little") == (a + b) % P
        hs.hs_fp_sub(ab, bb, r)
        assert int.from_bytes(bytes(r), "little") == (a - b) % P
    for _ in range(5):
        a = rng.randrange(1, P)
        r = out(48)
        hs.hs_fp_inv(buf(pr.fp_to_mont_bytes(a)), r)
        assert pr.fp_from_mont_bytes(bytes(r)) == pr.inv(a)
    # binary extended Euclid (single-thread tails): same inverse, 0 -> 0
    for a in [0, 1, 2, P - 1, P - 2, (P - 1) // 2, 1 << 380, (1 << 381) - 1] + [rng.randrange(1, P) for _ in range(200)]:
        r = out(48)
        hs.hs_fp_inv_vartime(buf(pr.fp_to_mont_bytes(a)), r)
        assert pr.fp_from_mont_bytes(bytes(r)) == (pr.inv(a) if a else 0), hex(a)


def f2b(a):
    return pr.fp_to_mont_bytes(a[0]) + pr.fp_to_mont_bytes(a[1])


def f2f(b):
    return (pr.fp_from_mont_bytes(b[:48]), pr.fp_from_mont_bytes(b[48:96]))


def test_fp2_rsqrt(hs):
    rng = random.Random(2)
    cases = [(rng.randrange(P), rng.randrange(P)) for _ in range(20)] + [(rng.randrange(P), 0) for _ in range(4)] + \
            [(0, rng.randrange(P)) for _ in range(4)] + [(4, 0), (P - 4, 0)]
    for a in cases:
        r = out(96)
        sq = hs.hs_fp2_rsqrt(buf(f2b(a)), r)
        assert bool(sq) == pr.f2_is_square(a)
        tgt = a if sq else pr.f2_mul(pr.SSWU_Z, a)
        assert pr.f2_mul(pr.f2_sqr(f2f(bytes(r))), tgt) == (1, 0)


def test_hash_to_g2_golden(hs):
    d = json.load(open(os.path.join(GOLD, "hash_to_g2_eth2.json")))
    dst = d["dst"].encode()
    for m, c, a in zip(d["msgs"], d["compressed"], d["affine"]):
        aff, comp = out(192), out(96)
        hs.hs_hash_to_g2(buf(bytes.fromhex(m)), C.c_size_t(32), buf(dst), C.c_uint32(len(dst)), aff, comp)
        assert bytes(aff).hex() == a and bytes(comp).hex() == c
    r = json.load(open(os.path.join(GOLD, "BLS12381G2_XMD_SHA-256_SSWU_RO_.json")))
    dst = r["dst"].encode()
    for v in r["vectors"]:
        m = v["msg"].encode()
        aff, comp = out(192), out(96)
        hs.hs_hash_to_g2(buf(m) if m else None, C.c_size_t(len(m)), buf(dst), C.c_uint32(len(dst)), aff, comp)
        x = tuple(int(t, 16) for t in v["P"]["x"].split(","))
        y = tuple(int(t, 16) for t in v["P"]["y"].split(","))
        assert pr.g2_from_mem(bytes(aff)) == (x, y)


def f12b(a):
    return b"".join(f2b(a[j][i]) for j in range(2) for i in range(3))


def f12f(b):
    c = [f2f(b[96 * k:96 * k + 96]) for k in range(6)]
    return ((c[0], c[1], c[2]), (c[3], c[4], c[5]))


def test_tower(hs):
    rng = random.Random(3)

    def rnd12():
        return tuple(tuple((rng.randrange(P), rng.randrange(P)) for _ in range(3)) for _ in range(2))
    for _ in range(2):
        a, b = rnd12(), rnd12()
        r = out(576)
        hs.hs_fp12_mul(buf(f12b(a)), buf(f12b(b)), r)
        assert f12f(bytes(r)) == pr.f12_mul(a, b)
        hs.hs_fp12_sqr(buf(f12b(a)), r)
        assert f12f(bytes(r)) == pr.f12_sqr(a)
        hs.hs_fp12_inv(buf(f12b(a)), r)
        assert f12f(bytes(r)) == pr.f12_inv(a)
        for n in (1, 2, 3):
            hs.hs_fp12_frob(buf(f12b(a)), n, r)
            assert f12f(bytes(r)) == pr.f12_frob(a, n)
        line = [(rng.randrange(P), rng.randrange(P)) for _ in range(3)]
        f = (C.c_uint8 * 576).from_buffer_copy(f12b(a))
        hs.hs_fp12_mul_by_line(f, buf(b"".join(f2b(x) for x in line)))
        assert f12f(bytes(f)) == pr.f12_mul(a, pr._line_sparse(*line))
        t = pr.f12_mul(pr.f12_conj(a), pr.f12_inv(a))
        t = pr.f12_mul(pr.f12_frob(t, 2), t)
        hs.hs_fp12_cyc_sqr(buf(f12b(t)), r)
        assert f12f(bytes(r)) == pr.f12_sqr(t)
        hs.hs_fp12_bytes(buf(f12b(a)), r)
        assert bytes(r) == pr.f12_to_bytes(a)
        hs.hs_final_exp(buf(f12b(a)), r)
        assert f12f(bytes(r)) == pr.final_exp(a)


@pytest.mark.parametrize("group,nseg", [(1, 1), (4, 8), (3, 5), (8, 63)])
def test_batch_pipeline_golden(hs, group, nseg):
    d = json.load(open(os.path.join(GOLD, "batch_scenarios.json")))
    for s in d["scenarios"]:
        raw = bytes.fromhex(s["sets"])
        sc = (C.c_uint64 * s["n"])(*[int(x) for x in s["scalars"]])
        gt = out(576)
        ok = hs.hs_batch_verify(buf(raw), C.c_size_t(s["n"]), sc, group, nseg, gt)
        assert bool(ok) == s["ok"], s["name"]
        if s["name"] != "infinite_pubkey":
            assert bytes(gt).hex() == s["gt"], s["name"]


def test_aggregate_golden(hs):
    a = json.load(open(os.path.join(GOLD, "aggregate.json")))
    pk, sg = bytes.fromhex(a["pubkeys"]), bytes.fromhex(a["signatures"])
    o1, o2 = out(96), out(192)
    hs.hs_aggregate_g1(buf(pk), C.c_size_t(len(pk) // 96), o1)
    hs.hs_aggregate_g2(buf(sg), C.c_size_t(len(sg) // 192), o2)
    assert bytes(o1).hex() == a["agg_pubkey"] and bytes(o2).hex() == a["agg_signature"]
    # doubling path: the same point twice
    hs.hs_aggregate_g1(buf(pk[:96] * 2), C.c_size_t(2), o1)
    assert pr.g1_from_mem(bytes(o1)) == pr.g1_mul(pr.g1_from_mem(pk[:96]), 2)


def test_subtract_all_golden(hs):
    """subtractAll (blst_min_pubkey_sig_core.nim:197-209) in the arrangement blsgpu_subtract_g1/_g2 launch."""
    a = json.load(open(os.path.join(GOLD, "aggregate.json")))
    pk, sg = bytes.fromhex(a["pubkeys"]), bytes.fromhex(a["signatures"])
    d1 = (C.c_uint8 * 96).from_buffer_copy(bytes.fromhex(a["agg_pubkey"]))
    d2 = (C.c_uint8 * 192).from_buffer_copy(bytes.fromhex(a["agg_signature"]))
    hs.hs_subtract_g1(d1, buf(pk), C.c_size_t(5))
    hs.hs_subtract_g2(d2, buf(sg), C.c_size_t(5))
    assert bytes(d1).hex() == a["sub5_pubkey"] and bytes(d2).hex() == a["sub5_signature"]
    # everything subtracted: infinity is the all-zero affine point; then infinity minus a point is its negative
    hs.hs_subtract_g1(d1, buf(pk[5 * 96:]), C.c_size_t(7))
    assert bytes(d1) == bytes(96)
    hs.hs_subtract_g1(d1, buf(pk[:96]), C.c_size_t(1))
    x, y = pr.g1_from_mem(pk[:96])
    assert pr.g1_from_mem(bytes(d1)) == (x, (-y) % pr.P)
    # dst equal to the only element: the doubling branch of the addition must not be taken for P + (-P)
    d1 = (C.c_uint8 * 96).from_buffer_copy(pk[:96])
    hs.hs_subtract_g1(d1, buf(pk[:96]), C.c_size_t(1))
    assert bytes(d1) == bytes(96)


def test_tail_programs(hs):
    """fpprog.hpp: the compiled warp-cooperative tail programs (final exponentiation of a product of partials, Horner
    over Miller-loop segments), executed round by round like k_fp_program, equal the straight-line formulas."""
    rng = random.Random(11)

    def rnd12():
        return tuple(tuple((rng.randrange(P), rng.randrange(P)) for _ in range(3)) for _ in range(2))
    stats = (C.c_int * 4)()
    for count in (1, 2, 3, 8):
        parts = [rnd12() for _ in range(count)]
        r = out(576)
        assert hs.hs_prog_final(buf(b"".join(f12b(x) for x in parts)), count, r, stats) == 1
        prod = parts[0]
        for x in parts[1:]:
            prod = pr.f12_mul(prod, x)
        assert f12f(bytes(r)) == pr.final_exp(prod), count
        assert stats[2] <= 1024 and stats[1] < 1400, list(stats)
        r2 = out(576)                           # the pair of programs around the external inversion (device path)
        assert hs.hs_prog_final_split(buf(b"".join(f12b(x) for x in parts)), count, r2, stats) == 1
        assert bytes(r2) == bytes(r), count
        assert stats[2] <= 1024 and stats[1] < 950, list(stats)
        assert stats[0] < 2600, list(stats)     # schedule length: 2 408-2 478 rounds (3 813 before the direct cyclotomic squaring)
    for nseg in (1, 2, 8, 21, 63):
        segs = b"".join(f12b(rnd12()) for _ in range(nseg))
        r, r2 = out(576), out(576)
        assert hs.hs_prog_combine(buf(segs), nseg, r, stats) == 1
        hs.hs_miller_combine(buf(segs), nseg, r2)
        assert bytes(r) == bytes(r2), nseg


def test_msm_horner_program(hs):
    """fpprog.hpp build_msm_horner_g1: the window Horner of the G1 MSM as a branch-free dataflow program over complete
    projective formulas == sum_w [2^(c w)] W_w computed by pyref, including infinite windows, equal and opposite
    points (the cases the Jacobian formulas of ec.cuh branch on)."""
    rng = random.Random(21)
    g = pr.G1_GEN
    stats = (C.c_int * 4)()

    def hom(pt):
        if pt is None:
            return (0, 1, 0)
        k = rng.randrange(1, P)
        return (pt[0] * k % P, pt[1] * k % P, k)
    cases = []
    for nwin, c in ((1, 5), (2, 3), (5, 13), (16, 16), (22, 12)):
        cases.append((nwin, c, [pr.g1_mul(g, rng.randrange(1, 1 << 64)) for _ in range(nwin)]))
    cases.append((4, 2, [None, None, None, None]))
    cases.append((4, 2, [pr.g1_mul(g, 7), None, None, None]))
    cases.append((3, 4, [None, pr.g1_mul(g, 5), None]))
    q = pr.g1_mul(g, 12345)
    cases.append((2, 1, [pr.g1_mul(q, 2), q]))                 # [2]q + [2]q: the addition must double
    cases.append((2, 1, [pr.g1_neg(pr.g1_mul(q, 2)), q]))      # [2]q - [2]q = infinity
    cases.append((3, 1, [q, pr.g1_neg(pr.g1_mul(q, 2)), q]))   # hits infinity in the middle, then adds again
    for nwin, c, ws in cases:
        exp = None
        for w in range(nwin - 1, -1, -1):
            if w != nwin - 1:
                exp = pr.g1_mul(exp, 1 << c) if exp is not None else None
            exp = pr.g1_add(exp, ws[w])
        inp = b"".join(pr.fp_to_mont_bytes(v) for pt in ws for v in hom(pt))
        r = out(3 * 48)
        assert hs.hs_prog_msm_horner(buf(inp), nwin, c, r, stats) == 1
        o = [pr.fp_from_mont_bytes(bytes(r)[48 * i:48 * i + 48]) for i in range(3)]
        if exp is None:
            assert o[2] == 0 and o[1] != 0, (nwin, c)
        else:
            zi = pr.inv(o[2])
            assert (o[0] * zi % P, o[1] * zi % P) == exp, (nwin, c)
        assert stats[2] <= 1024, list(stats)


def _g2_hom_bytes(pt, rng):
    """affine G2 point (or None) -> 6 Montgomery fp of a random homogeneous representative"""
    if pt is None:
        x, y, z = (0, 0), (rng.randrange(1, P), rng.randrange(P)), (0, 0)
    else:
        k = (rng.randrange(1, P), rng.randrange(P))
        x, y, z = pr.f2_mul(pt[0], k), pr.f2_mul(pt[1], k), k
    return b"".join(pr.fp_to_mont_bytes(c) for v in (x, y, z) for c in v)


def _g2_from_hom(raw):
    v = [pr.fp_from_mont_bytes(raw[48 * i:48 * i + 48]) for i in range(6)]
    z = (v[4], v[5])
    if z == (0, 0):
        return None
    zi = pr.f2_inv(z)
    return pr.f2_mul((v[0], v[1]), zi), pr.f2_mul((v[2], v[3]), zi)


def test_g2_programs(hs):
    """fpprog.hpp build_g2_clear_cofactor / build_g2_mul64 (complete projective formulas on the twist, one warp per set
    on the device) against pyref: cofactor clearing of points on E2 outside the subgroup, 64-bit multiples incl. edge
    scalars, the point at infinity."""
    rng = random.Random(33)
    stats = (C.c_int * 4)()
    # points on E2 (not in G2): x random, y = sqrt(x^3 + 4(1+u))
    pts = []
    while len(pts) < 3:
        x = (rng.randrange(P), rng.randrange(P))
        rhs = pr.f2_add(pr.f2_mul(pr.f2_sqr(x), x), (4, 4))
        if pr.f2_is_square(rhs):
            pts.append((x, pr.f2_sqrt(rhs)))
    for pt in pts + [None]:
        r = out(6 * 48)
        assert hs.hs_prog_g2_clear_cofactor(buf(_g2_hom_bytes(pt, rng)), r, stats) == 1
        exp = pr.g2_clear_cofactor(pt) if pt is not None else None
        assert _g2_from_hom(bytes(r)) == exp
        assert stats[2] <= 1024, list(stats)
    g = pr.G2_GEN
    q = pr.g2_mul(g, 987654321)
    for k in [1, 2, 3, 0x8000000000000000, 0xffffffffffffffff, 0x5555555555555555] + [rng.getrandbits(64) for _ in range(4)]:
        r = out(6 * 48)
        assert hs.hs_prog_g2_mul64(buf(_g2_hom_bytes(q, rng)), C.c_uint64(k), r, stats) == 1
        assert _g2_from_hom(bytes(r)) == pr.g2_mul(q, k), hex(k)
    r = out(6 * 48)
    assert hs.hs_prog_g2_mul64(buf(_g2_hom_bytes(None, rng)), C.c_uint64(12345), r, stats) == 1
    assert _g2_from_hom(bytes(r)) is None
    assert stats[2] <= 1024, list(stats)


def test_fp12_product_program(hs):
    """build_fp12_product (GT product of a segment row in small batches) == the product by pyref."""
    rng = random.Random(66)
    stats = (C.c_int * 4)()
    for count in (1, 2, 3, 5, 8, 16):
        vals = [tuple(tuple((rng.randrange(P), rng.randrange(P)) for _ in range(3)) for _ in range(2)) for _ in range(count)]
        r = out(576)
        assert hs.hs_prog_fp12_product(buf(b"".join(f12b(x) for x in vals)), count, r, stats) == 1
        prod = vals[0]
        for x in vals[1:]:
            prod = pr.f12_mul(prod, x)
        assert f12f(bytes(r)) == prod, count
        assert stats[2] <= 1024, (count, list(stats))


def test_msm_horner_program_g2(hs):
    """build_msm_horner_g2 (window Horner of the signature-side MSM) == sum_w [2^(c w)] W_w by pyref, with an infinite
    window and the 64-bit shape the batch verifier uses (5 windows of 13 bits)."""
    rng = random.Random(55)
    stats = (C.c_int * 4)()
    g = pr.G2_GEN
    for nwin, c, holes in ((5, 13, ()), (3, 4, (1,)), (1, 7, ())):
        ws = [None if w in holes else pr.g2_mul(g, rng.randrange(1, 1 << 64)) for w in range(nwin)]
        exp = None
        for w in range(nwin - 1, -1, -1):
            if w != nwin - 1 and exp is not None:
                exp = pr.g2_mul(exp, 1 << c)
            exp = pr.g2_add(exp, ws[w])
        inp = b"".join(_g2_hom_bytes(pt, rng) for pt in ws)
        r = out(6 * 48)
        assert hs.hs_prog_msm_horner_g2(buf(inp), nwin, c, r, stats) == 1
        assert _g2_from_hom(bytes(r)) == exp, (nwin, c)


def test_miller_lines_program(hs):
    """fpprog.hpp build_miller_lines == pairing.cuh miller_lines, word for word (every Fp value is canonical, so equal
    formulas give equal bits): 68 line triples of a pair, for several (Q, P)."""
    rng = random.Random(44)
    stats = (C.c_int * 4)()
    for _ in range(3):
        q = pr.g2_mul(pr.G2_GEN, rng.randrange(1, 1 << 200))
        pt = pr.g1_mul(pr.G1_GEN, rng.randrange(1, 1 << 200))
        o1, o2 = out(68 * 6 * 48), out(68 * 72 * 4)
        assert hs.hs_prog_miller_lines(buf(pr.g2_to_mem(q)), buf(pr.g1_to_mem(pt)), o1, o2, stats) == 1
        assert bytes(o1) == bytes(o2)
        assert stats[2] <= 1024, list(stats)


def test_g1_mul_windowed(hs):
    """pt_mul_u64_w4 (signed 4-bit windows) == pt_mul_u64 (double-and-add) == pyref, incl. edge scalars and infinity."""
    rng = random.Random(5)
    a = json.load(open(os.path.join(GOLD, "aggregate.json")))
    pk = bytes.fromhex(a["pubkeys"])[:96]
    pt = pr.g1_from_mem(pk)
    ks = [1, 2, 8, 9, 15, 16, 0x8888888888888888, 0x9999999999999999, 0xffffffffffffffff, 0x7777777777777777, 0] + \
         [rng.getrandbits(64) for _ in range(12)]
    for k in ks:
        o1, o2 = out(96), out(96)
        hs.hs_g1_mul_u64_w4(buf(pk), C.c_uint64(k), o1)
        hs.hs_g1_mul_u64(buf(pk), C.c_uint64(k), o2)
        assert bytes(o1) == bytes(o2), hex(k)
        if k:
            assert pr.g1_from_mem(bytes(o1)) == pr.g1_mul(pt, k), hex(k)
    o1 = out(96)
    hs.hs_g1_mul_u64_w4(buf(bytes(96)), C.c_uint64(12345), o1)
    assert bytes(o1) == bytes(96)


def test_from_bytes_with_checks(hs):
    """io.cuh on the host against pyref's restatement of BLST's fromBytes (error code and point): every exit of
    uncompress / deserialize, infinity rule, subgroup tests.  The cases start from BLST's keys and signatures in
    aggregate.json."""
    rng = random.Random(11)
    a = json.load(open(os.path.join(GOLD, "aggregate.json")))
    pks, sigs = bytes.fromhex(a["pubkeys"]), bytes.fromhex(a["signatures"])
    g1_cases = [pr.g1_compress(pr.g1_from_mem(pks[96 * i:96 * i + 96])) for i in range(3)]
    good = g1_cases[0]
    g1_cases += [bytes([good[0] ^ 0x20]) + good[1:], bytes([good[0] & 0x7f]) + good[1:], bytes([0xc0]) + bytes(47),
                 bytes([0xc0]) + bytes(46) + b"\x01", bytes([0x80 | 0x1a]) + P.to_bytes(48, "big")[1:],
                 bytes([0x80]) + bytes(47)]
    g1_cases += [bytes([0x80]) + x.to_bytes(47, "big") for x in range(1, 12)]
    g1_cases += [pr.g1_serialize(pr.g1_from_mem(pks[:96])), bytes([0x40]) + bytes(95), bytes(96), good + bytes(48)]
    seen = set()
    for c in g1_cases:
        for gc in (1, 0):
            o = out(96)
            err = hs.hs_pubkey_from_bytes(buf(c), len(c), gc, o)
            assert (err, bytes(o)) == pr.pubkey_from_bytes(c, group_check=bool(gc)), (c.hex(), gc)
            seen.add(err)
    assert seen >= {0, 1, 2, 3, 6}
    o = out(48)
    hs.hs_g1_compress(buf(pks[:96]), o)
    assert bytes(o) == good
    g2_cases = [pr.g2_compress(pr.g2_from_mem(sigs[192 * i:192 * i + 192])) for i in range(3)]
    good = g2_cases[0]
    g2_cases += [bytes([good[0] ^ 0x20]) + good[1:], bytes([0xc0]) + bytes(95), good[:48] + P.to_bytes(48, "big"),
                 bytes([0x80]) + bytes(95), pr.g2_serialize(pr.g2_from_mem(sigs[:192])), bytes(192),
                 bytes([0x40]) + bytes(191)]
    for _ in range(8):
        b = bytearray(rng.randrange(P).to_bytes(48, "big") + rng.randrange(P).to_bytes(48, "big"))
        b[0] = (b[0] & 0x1f) | 0x80
        g2_cases.append(bytes(b))
    seen = set()
    for c in g2_cases:
        for gc in (1, 0):
            o = out(192)
            err = hs.hs_signature_from_bytes(buf(c), len(c), gc, o)
            assert (err, bytes(o)) == pr.signature_from_bytes(c, group_check=bool(gc)), (c.hex(), gc)
            seen.add(err)
    assert seen >= {0, 1, 2, 3}


def test_programs_in_the_lincomb_format_too(hs):
    """Format 2 of the programs (rounds of products and rounds of linear combinations, fpprog.hpp compile2 / fplin.cuh;
    BLSGPU_PROG_FORMAT=2 on the device — measured slower there, so format 1 is the default): every program test above
    runs again in format 2, and the flattening is checked to shorten the schedules."""
    stats1, stats2 = (C.c_int * 4)(), (C.c_int * 4)()
    rng = random.Random(5)

    def rnd12():
        return tuple(tuple((rng.randrange(P), rng.randrange(P)) for _ in range(3)) for _ in range(2))
    part = buf(f12b(rnd12()))
    r1, r2 = out(576), out(576)
    hs.hs_set_program_format(1)
    assert hs.hs_prog_final_split(part, 1, r1, stats1) == 1
    hs.hs_set_program_format(2)
    try:
        assert hs.hs_prog_final_split(part, 1, r2, stats2) == 1
        test_tail_programs(hs)
        test_msm_horner_program(hs)
        test_g2_programs(hs)
        test_fp12_product_program(hs)
        test_msm_horner_program_g2(hs)
        test_miller_lines_program(hs)
    finally:
        hs.hs_set_program_format(0)
    assert bytes(r1) == bytes(r2)
    assert stats2[0] < 1100 and stats1[0] > 2 * stats2[0], (list(stats1), list(stats2))   # 2 408 -> 973 rounds
    assert stats2[1] == stats1[1]                                                           # same multiplication rounds
