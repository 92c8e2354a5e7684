"""CPU: pin the oracle.  (1) the pure-Python restatement (oracle/pyref.py) against the reference's own RFC 9380
known-answer vectors; (2) pyref and the BLST build (oracle/_ref) against the fixtures produced by running BLST on
the tests/t_batch_verifier.nim scenarios (tools/gen_golden.py)."""
import hashlib
import json
import os

import pytest

from oracle import pyref as pr

GOLD = os.path.join(os.path.dirname(__file__), "golden")


def load(name):
    return json.load(open(os.path.join(GOLD, name)))


@pytest.mark.parametrize("fname", ["expand_message_xmd_SHA256_38.json", "expand_message_xmd_SHA256_256.json"])
def test_expand_message_xmd_vectors(fname):
    d = load(fname)
    dst = d["DST"].encode()
    for v in d["tests"]:
        out = pr.expand_message_xmd(v["msg"].encode(), dst, int(v["len_in_bytes"], 16))
        assert out.hex() == v["uniform_bytes"]


def test_hash_to_curve_g2_vectors():
    d = load("BLS12381G2_XMD_SHA-256_SSWU_RO_.json")
    dst = d["dst"].encode()

    def f2(s):
        return tuple(int(t, 16) for t in s.split(","))
    for v in d["vectors"]:
        m = v["msg"].encode()
        u = pr.hash_to_field_fp2(m, dst)
        assert list(u) == [f2(x) for x in v["u"]]
        q0 = pr.iso3_g2(pr.sswu_g2(u[0]))
        q1 = pr.iso3_g2(pr.sswu_g2(u[1]))
        assert q0 == (f2(v["Q0"]["x"]), f2(v["Q0"]["y"]))
        assert q1 == (f2(v["Q1"]["x"]), f2(v["Q1"]["y"]))
        assert pr.hash_to_g2(m, dst) == (f2(v["P"]["x"]), f2(v["P"]["y"]))


def parse_sets(raw):
    return [(pr.g1_from_mem(raw[i:i + 96]), raw[i + 96:i + 128], pr.g2_from_mem(raw[i + 128:i + 320]))
            for i in range(0, len(raw), 320)]


def test_pyref_matches_blst_batch_fixtures():
    d = load("batch_scenarios.json")
    srb = bytes.fromhex(d["srb"])
    seen = 0
    for s in d["scenarios"]:
        if s["n"] > 4 and s["name"] not in ("valid_15",):
            continue                                    # pure Python: keep the CPU suite short
        raw = bytes.fromhex(s["sets"])
        assert [str(x) for x in pr.rlc_scalars(srb, s["n"], s["chunks"])] == s["scalars"]
        ok, gt = pr.batch_verify(parse_sets(raw), srb, s["chunks"])
        assert ok == s["ok"], s["name"]
        if s["name"] != "infinite_pubkey":
            assert gt.hex() == s["gt"], s["name"]
        seen += 1
    assert seen >= 8


def test_pyref_hash_to_g2_eth2_fixture():
    d = load("hash_to_g2_eth2.json")
    for m, c, a in zip(d["msgs"], d["compressed"], d["affine"]):
        h = pr.hash_to_g2(bytes.fromhex(m), d["dst"].encode())
        assert pr.g2_compress(h).hex() == c and pr.g2_to_mem(h).hex() == a


def test_pyref_msm_and_aggregate_fixtures():
    d = load("msm_g1.json")
    for c in d["cases"][:3]:
        pts, sc = bytes.fromhex(c["points"]), bytes.fromhex(c["scalars"])
        acc = None
        for i in range(c["n"]):
            k = int.from_bytes(sc[32 * i:32 * i + 32], "little") & ((1 << c["nbits"]) - 1)
            acc = pr.g1_add(acc, pr.g1_mul(pr.g1_from_mem(pts[96 * i:96 * i + 96]), k))
        assert pr.g1_to_mem(acc).hex() == c["result"]
    a = load("aggregate.json")
    pk = bytes.fromhex(a["pubkeys"])
    acc = None
    for i in range(0, len(pk), 96):
        acc = pr.g1_add(acc, pr.g1_from_mem(pk[i:i + 96]))
    assert pr.g1_to_mem(acc).hex() == a["agg_pubkey"]


def test_final_exp_power_identity():
    # hard part used by the device code: (z-1)^2 (z+p)(z^2+p^2-1) + 3 == 3 (p^4-p^2+1)/r  (pairing.c:371-404)
    assert pr.HARD_POWER == 3 * (pr.P ** 4 - pr.P ** 2 + 1) // pr.R_ORDER
    assert pr.FINAL_EXP_POWER == (pr.P ** 6 - 1) * (pr.P ** 2 + 1) * pr.HARD_POWER


# ---- the real reference (BLST build) against the same fixtures ----------------------------------------------
def _blst():
    try:
        from oracle import blst_ref
        return blst_ref
    except Exception as e:          # not built on this machine
        pytest.skip(f"oracle/_ref not built: {e}")


def test_blst_reproduces_batch_fixtures():
    br = _blst()
    d = load("batch_scenarios.json")
    srb = bytes.fromhex(d["srb"])
    for s in d["scenarios"]:
        ok, gt = br.batch_verify(bytes.fromhex(s["sets"]), srb, s["chunks"])
        assert ok == s["ok"] and gt.hex() == s["gt"], s["name"]
        assert [str(x) for x in br.rlc_scalars(srb, s["n"], s["chunks"])] == s["scalars"]


def test_blst_mt_replica_and_rank_decomposition():
    br = _blst()
    srb = hashlib.sha256(b"Mr F was here").digest()
    sets = br.make_sets(0, 21)
    assert br.batch_verify_mt(sets, srb, 4) is True
    bad = bytearray(sets)
    bad[7 * 320 + 128:8 * 320] = sets[128:320]
    assert br.batch_verify_mt(bytes(bad), srb, 4) is False
    for s in (sets, bytes(bad)):
        ok, gt = br.batch_verify(s, srb, 4)
        parts = b"".join(br.partial(s[f * 320:(f + c) * 320], f, 21, srb, 4)[0] for f, c in ((0, 7), (7, 7), (14, 7)))
        assert br.finalize(parts) == (ok, gt)


def test_blst_hash_to_g2_rfc_vectors():
    br = _blst()
    d = load("BLS12381G2_XMD_SHA-256_SSWU_RO_.json")
    dst = d["dst"].encode()
    for v in d["vectors"]:
        m = v["msg"].encode()
        if not m:
            continue
        _, aff = br.hash_to_g2(m, len(m), dst)
        x = tuple(int(t, 16) for t in v["P"]["x"].split(","))
        y = tuple(int(t, 16) for t in v["P"]["y"].split(","))
        assert pr.g2_from_mem(aff) == (x, y)


# ---- the stand-in used when oracle/_ref is not built: its stored answers against pyref --------------------------
def test_replay_table_matches_pyref(monkeypatch):
    """A sample of every kind of entry in tests/golden/oracle_answers.json.gz, on the inputs the GPU tests make (here
    rebuilt with pyref instead of the library), recomputed with pyref."""
    import random
    from oracle import replay as rp
    monkeypatch.setattr(rp, "INPUTS_ON_DEVICE", False)
    srb = hashlib.sha256(b"Mr F was here").digest()

    def same(name, args, ref):
        assert rp._answer(name, args, None) == ref, name
    for n, chunks in ((1, 0), (2, 4)):                                   # test_valid_batches
        sets = rp.make_sets(0, n, b"msg")
        same("batch_verify", (sets, srb, chunks, None), rp._ref_batch_verify(sets, srb, chunks, None))
    s1, s2 = rp.make_set(1, b"msg1"), rp.make_set(2, b"msg2")            # test_wrong_signature
    bad = s1 + s2[:128] + s1[128:]
    same("batch_verify", (bad, srb, 0, None), rp._ref_batch_verify(bad, srb, 0, None))
    pts, sc = rp.msm_points(0xFACADE, 3)                                 # test_msm_g1_255[3]
    same("msm_g1", (pts, sc, 255), rp._ref_msm(pts, sc, 255, False))
    sets = rp.make_sets(3, 2)                                            # test_msm_g2[2-64]
    g2 = b"".join(sets[i * 320 + 128:(i + 1) * 320] for i in range(2))
    rng = random.Random(2 * 1000 + 64)
    sc2 = b"".join(rng.getrandbits(64).to_bytes(8, "little") for _ in range(2))
    same("msm_g2", (g2, sc2, 64), rp._ref_msm(g2, sc2, 64, True))
    dst = pr.DST_ETH2                                                    # test_hash_to_g2_eth2_dst
    msgs = b"".join(hashlib.sha256(b"m%d" % i).digest() for i in range(300))
    same("hash_to_g2", (msgs, 32, dst), rp._ref_hash_to_g2(msgs, 32, dst))
    sets = [rp.make_set(i, b"same message") for i in range(2)]           # test_combine_same_message[2]
    pks, sigs = b"".join(s[:96] for s in sets), b"".join(s[128:] for s in sets)
    same("combine", (srb, pks, sigs), rp._ref_combine(srb, pks, sigs))
    rng = random.Random(1)                                               # test_aggregate_verify[1]
    m = [bytes(rng.randrange(256) for _ in range(rng.choice([0, 1, 31, 32, 33, 55, 56, 64, 101])))]
    pk, sig = rp.sign(900, m[0])
    agg = rp.aggregate_g2(sig)[1]
    for args in ((pk, m, agg, dst), (bytes(96), m, agg, dst), (pk, m, bytes(192), dst)):
        same("aggregate_verify", args, rp._ref_aggregate_verify(*args))
    h = hashlib.sha256(b"sync committee 2").digest()                     # test_fast_aggregate_verify[2]
    member, aset = rp.fast_aggregate_set(3000, 2, h)
    for args in ((member, h, aset[128:], dst), (member[:-96], h, aset[128:], dst)):
        same("fast_aggregate_verify", args, rp._ref_fast_aggregate_verify(*args))
