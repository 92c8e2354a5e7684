"""GPU: batch verification of compressed signature sets (blsgpu_batch_verify_compressed): the signatures are decoded and
subgroup-checked inside the pipeline.  A batch of valid encodings must give exactly what blsgpu_batch_verify gives on the
decoded 320-byte sets, at every route boundary; a bad encoding must fail the batch with an all-zero GT and report
Signature.fromBytes' status at its index; multi-device shares and CUDA-graph replays must do the same."""
import ctypes as C
import json
import os
import random

import pytest

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden")
P = 0x1a0111ea397fe69a4b1ba7b6434bacd764774b84f38512bf6730d2a0f6b0f6241eabfffeb153ffffb9feffffffffaaab
ZERO_GT = bytes(576)


@pytest.fixture(scope="module")
def big():
    import nim_blscurve_b200 as bg
    c = bg.BatchedBLSVerifierCache(max_sets=40001, device=0)
    yield c
    c.close()


def compress(cache, sets320):
    """224-byte records: key and message of each 320-byte set, its signature compressed on the device."""
    import nim_blscurve_b200 as bg
    n = len(sets320) // 320
    sigs = b"".join(sets320[320 * i + 128:320 * i + 320] for i in range(n))
    comp = bg.signaturesToBytes(cache, sigs)
    return b"".join(sets320[320 * i:320 * i + 128] + comp[96 * i:96 * i + 96] for i in range(n))


def device_sets(cache, seed, n):
    import nim_blscurve_b200 as bg
    out = (C.c_uint8 * (320 * n))()
    assert bg.lib().blsgpu_make_sets(cache.handle, seed, 0, n, out, 0) == 0
    return bytes(out)


def with_sig(recs, i, sig96):
    return recs[:224 * i + 128] + sig96 + recs[224 * i + 224:]


def with_sig320(sets, i, sig192):
    return sets[:320 * i + 128] + sig192 + sets[320 * i + 320:]


def test_golden_scenarios_compressed(big, br):
    """Every scenario of batch_scenarios.json with its signatures compressed: BLST's stored verdict and GT, with the
    derived scalars and with the explicit ones."""
    d = json.load(open(os.path.join(GOLD, "batch_scenarios.json")))
    srb = bytes.fromhex(d["srb"])
    for s in d["scenarios"]:
        sets = bytes.fromhex(s["sets"])
        recs = compress(big, sets)
        want_st = [br.signature_from_bytes(recs[224 * i + 128:224 * i + 224])[0] for i in range(len(recs) // 224)]
        ok, st, gt = big.verify_compressed_raw(recs, srb, s["chunks"], want_gt=True)
        assert st == want_st, s["name"]
        if any(want_st):                                     # a signature outside G2 fails the batch
            assert (ok, gt) == (False, ZERO_GT), s["name"]
        elif s["name"] != "infinite_pubkey":
            assert (ok, gt.hex()) == (s["ok"], s["gt"]), s["name"]
        else:
            assert (ok, gt) == (False, ZERO_GT)
        ok2, st2, gt2 = big.verify_compressed_raw(recs, srb, 0, scalars=[int(x) for x in s["scalars"]], want_gt=True)
        assert (ok2, st2, gt2) == (ok, st, gt), s["name"]


SIZES = [1, 2, 64, 129, 1025, 3000, 4600, 9000, 40001]


@pytest.mark.parametrize("n", SIZES)
def test_valid_and_swapped_match_the_decoded_path(big, br, srb, n):
    """Valid batches, and batches with two signatures swapped (valid encodings, wrong sets), give the verdict and GT of
    blsgpu_batch_verify on the decoded sets, with every status 0."""
    sets = br.make_sets(4000 + n, n) if n <= 2 else device_sets(big, 11 + n, n)
    recs = compress(big, sets)
    chunks = 0 if n < 3 else 8
    ok, st, gt = big.verify_compressed_raw(recs, srb, chunks, want_gt=True)
    assert (ok, gt) == big.verify_raw(sets, srb, chunks, want_gt=True) and ok is True
    assert st == [0] * n
    if n == 1:
        return
    j = n // 2
    sw = with_sig320(with_sig320(sets, 0, sets[320 * j + 128:320 * j + 320]), j, sets[128:320])
    swr = with_sig(with_sig(recs, 0, recs[224 * j + 128:224 * j + 224]), j, recs[128:224])
    ok, st, gt = big.verify_compressed_raw(swr, srb, chunks, want_gt=True)
    assert ok is False and gt != ZERO_GT and st == [0] * n
    assert (ok, gt) == big.verify_raw(sw, srb, chunks, want_gt=True)


def encodings(br):
    """The 36 encodings of test_signatures_from_bytes: valid points of other sets, the other root, bad flags, infinity
    with and without garbage, x >= p, x == 0, random x on and off the curve (none in G2)."""
    rng = random.Random(6)
    sets = br.make_sets(700, 10)
    cases = [br.g2_compress(sets[320 * i + 128:320 * i + 320]) for i in range(10)]
    good = cases[0]
    cases.append(bytes([good[0] ^ 0x20]) + good[1:])
    cases.append(bytes([good[0] & 0x7f]) + good[1:])
    cases.append(bytes([0xc0]) + bytes(95))
    cases.append(bytes([0xc0]) + bytes(94) + b"\x01")
    cases.append(bytes([0x80 | 0x1a]) + P.to_bytes(48, "big")[1:] + bytes(48))
    cases.append(good[:48] + P.to_bytes(48, "big"))
    cases.append(bytes([0x80]) + bytes(95))
    while len(cases) < 36:
        xi, xr = rng.randrange(P), rng.randrange(P)
        b = bytearray(xi.to_bytes(48, "big") + xr.to_bytes(48, "big"))
        b[0] = (b[0] & 0x1f) | 0x80 | (0x20 if rng.random() < 0.5 else 0)
        cases.append(bytes(b))
    return cases


@pytest.mark.parametrize("n", [129, 3000, 9000])
def test_each_encoding_at_first_middle_last(big, br, srb, n):
    """One encoding at a time at the first, a middle and the last index: status = Signature.fromBytes' status there and
    0 elsewhere; a failing status fails the batch with an all-zero GT; a decodable one (other set's signature, the other
    root, infinity) gives the decoded path's verdict and GT."""
    cases = encodings(br)
    want = [br.signature_from_bytes(c) for c in cases]
    assert {w[0] for w in want} >= {0, 1, 2, 3}
    sets = device_sets(big, 300 + n, n)
    recs = compress(big, sets)
    for idx in (0, n // 2, n - 1):
        for c, (code, point) in zip(cases, want):
            ok, st, gt = big.verify_compressed_raw(with_sig(recs, idx, c), srb, 4, want_gt=True)
            exp = [0] * n
            exp[idx] = code
            assert st == exp, (idx, c.hex()[:8])
            if code:
                assert (ok, gt) == (False, ZERO_GT), (idx, code)
            else:
                assert (ok, gt) == big.verify_raw(with_sig320(sets, idx, point), srb, 4, want_gt=True), (idx, c.hex()[:8])


def test_multi_device_shares(br, srb):
    """Device 0 listed twice: a bad signature in either share gives the one-device statuses and 0; a valid batch gives
    the one-device verdict and GT."""
    import nim_blscurve_b200 as bg
    n = 301
    one = bg.BatchedBLSVerifierCache(max_sets=n, device=0)
    two = bg.BatchedBLSVerifierCache(max_sets=n, devices=[0, 0])
    try:
        sets = device_sets(one, 77, n)
        recs = compress(one, sets)
        r1, r2 = one.verify_compressed_raw(recs, srb, 4, want_gt=True), two.verify_compressed_raw(recs, srb, 4, want_gt=True)
        assert r1 == r2 and r1[0] is True
        bad_curve = bytes([0x80]) + bytes(95)                              # x == 0: not on the curve
        not_g2 = next(c for c in encodings(br) if br.signature_from_bytes(c)[0] == 3)
        for idx, c in ((10, bad_curve), (250, not_g2), (150, bad_curve)):
            r1 = one.verify_compressed_raw(with_sig(recs, idx, c), srb, 4, want_gt=True)
            r2 = two.verify_compressed_raw(with_sig(recs, idx, c), srb, 4, want_gt=True)
            assert r1 == r2 and r1[0] is False and r1[2] == ZERO_GT
            assert r1[1][idx] == br.signature_from_bytes(c)[0] and sum(1 for x in r1[1] if x) == 1
    finally:
        one.close()
        two.close()


def test_graph_replay_is_fresh(br, srb):
    """129 sets from one host buffer: direct call, capture, replay with a changing srb and a bad signature at the third
    call; then a valid replay again.  Interleaved 320-byte calls of the same size keep their own graph."""
    import hashlib
    import nim_blscurve_b200 as bg
    n = 129
    c = bg.BatchedBLSVerifierCache(max_sets=n, device=0)
    try:
        sets = device_sets(c, 5, n)
        recs = compress(c, sets)
        bad = with_sig(recs, 40, bytes([0xc0]) + bytes(94) + b"\x01")
        srbs = [hashlib.sha256(bytes([k])).digest() for k in range(6)]
        for k, (r, code) in enumerate(((recs, 0), (recs, 0), (bad, 1), (recs, 0), (bad, 1), (recs, 0))):
            ok, st, gt = c.verify_compressed_raw(r, srbs[k], 8, want_gt=True)
            assert st[40] == code and sum(1 for x in st if x) == (1 if code else 0), k
            if code:
                assert (ok, gt) == (False, ZERO_GT), k
            else:
                assert (ok, gt) == c.verify_raw(sets, srbs[k], 8, want_gt=True) and ok is True, k
        # the graph replays (one launch) at the later calls
        c.verify_compressed_raw(recs, srbs[0], 8)
        assert bg.lib().blsgpu_last_launches(c.handle) == 1
    finally:
        c.close()


def test_empty_and_argument_errors(big, srb):
    import nim_blscurve_b200 as bg
    L = bg.lib()
    gt = (C.c_uint8 * 576)(*([7] * 576))
    assert L.blsgpu_batch_verify_compressed(big.handle, None, 0, srb, 0, None, gt, None) == 0 and bytes(gt) == ZERO_GT
    assert L.blsgpu_batch_verify_compressed(big.handle, None, 3, srb, 0, None, None, None) == -2
    assert L.blsgpu_batch_verify_compressed(big.handle, bytes(224 * 40002), 40002, srb, 0, None, None, None) == -3
    sc = (C.c_uint64 * 2)(5, 0)
    assert L.blsgpu_batch_verify_compressed(big.handle, bytes(448), 2, srb, 0, sc, None, None) == -2
    assert bg.batchVerifyCompressed(bg.Taskpool(4), big, [], srb) == (False, [])
