"""GPU: (1) the CUDA path against the committed golden fixtures (outputs of the reference's BLST build,
tests/golden/*.json) — no oracle needed at run time; (2) the rank decomposition on one device: shares computed
by blsgpu_partial and combined by blsgpu_finalize must reproduce the single-call verdict and GT; (3) size-
independent properties at a larger size."""
import ctypes as C
import hashlib
import json
import os

import pytest

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden")


def load(name):
    return json.load(open(os.path.join(GOLD, name)))


def test_batch_scenarios_golden(cache):
    d = load("batch_scenarios.json")
    srb = bytes.fromhex(d["srb"])
    for s in d["scenarios"]:
        ok, gt = cache.verify_raw(bytes.fromhex(s["sets"]), srb, s["chunks"], want_gt=True)
        assert ok == s["ok"], s["name"]
        if s["name"] != "infinite_pubkey":
            assert gt.hex() == s["gt"], s["name"]
        # explicit scalars must reproduce the same GT
        ok2, gt2 = cache.verify_raw(bytes.fromhex(s["sets"]), srb, 0, scalars=[int(x) for x in s["scalars"]], want_gt=True)
        assert (ok2, gt2) == (ok, gt)


def test_hash_msm_aggregate_golden(cache):
    import nim_blscurve_b200 as bg
    d = load("hash_to_g2_eth2.json")
    comp, aff = bg.hashToG2(cache, b"".join(bytes.fromhex(m) for m in d["msgs"]), 32, d["dst"].encode())
    assert comp.hex() == "".join(d["compressed"]) and aff.hex() == "".join(d["affine"])
    for c in load("msm_g1.json")["cases"]:
        assert bg.msmG1(cache, bytes.fromhex(c["points"]), bytes.fromhex(c["scalars"]), c["nbits"]).hex() == c["result"]
    a = load("aggregate.json")
    pk, sg = bytes.fromhex(a["pubkeys"]), bytes.fromhex(a["signatures"])
    assert bg.aggregateAll(cache, [pk[i:i + 96] for i in range(0, len(pk), 96)]) == (True, bytes.fromhex(a["agg_pubkey"]))
    assert bg.aggregateAll(cache, [sg[i:i + 192] for i in range(0, len(sg), 192)]) == (True, bytes.fromhex(a["agg_signature"]))


@pytest.mark.parametrize("world", [2, 3, 8])
def test_rank_shares_on_one_device(cache, br, srb, world):
    import nim_blscurve_b200 as bg
    be = bg.GpuBackend(cache)
    sets = br.make_sets(0, 21)
    bad = bytearray(sets)
    bad[13 * 320 + 128:14 * 320] = sets[128:320]
    for s in (sets, bytes(bad)):
        for chunks in (0, 5):
            ok, gt = br.batch_verify(s, srb, chunks)
            parts, flags = b"", 0
            for r in range(world):
                first, cnt = bg.shard_range(21, world, r)
                p, f = be.partial(s[first * 320:(first + cnt) * 320], first, 21, srb, chunks)
                parts += p
                flags |= f
            assert flags == 0
            assert be.finalize(parts) == (ok, gt)
            # mixing GPU partials with BLST partials is still exact after the final exponentiation
            first, cnt = bg.shard_range(21, world, 0)
            mixed = br.partial(s[:cnt * 320], 0, 21, srb, chunks)[0] + parts[576:]
            assert be.finalize(mixed) == (ok, gt)
    # empty share -> neutral partial ; infinite pubkey -> flag
    p, f = be.partial(b"", 0, 21, srb, 4)
    assert be.finalize(p) == (True, br.finalize(br.partial(b"", 0, 21, srb, 4)[0])[1])
    inf = bytes(96) + sets[96:320]
    p_inf, f_inf = be.partial(inf, 0, 1, srb, 0)
    assert f_inf != 0
    # ... and the flagged share's partial is sealed: zero absorbs the product, the final exponentiation keeps it zero,
    # so the 576 bytes alone carry the verdict (bls_batch_verifier.nim:153: update() false -> batch false)
    assert p_inf == bytes(576)
    good = be.partial(sets[:320 * 5], 0, 5, srb, 0)[0]
    assert be.finalize(good + p_inf) == (False, bytes(576))


def test_deferred_signature_pair_vs_blst(br, srb):
    """Large batch behind long scalar chains (the drop-in's tp.numThreads = 4 chunks of 4 100 sets): the n set pairs run
    their multi-Miller loop without waiting for the signature-side MSM, pair number n = (S, -G1) gets its own loop and
    the two values are multiplied (blsgpu.cu run_partial).  Verdict and GT must equal BLST's."""
    import nim_blscurve_b200 as bg
    n = 16400
    big = bg.BatchedBLSVerifierCache(max_sets=n, device=0)
    try:
        out = (C.c_uint8 * (320 * n))()
        assert bg.lib().blsgpu_make_sets(big.handle, 5, 0, n, out, 0) == 0
        sets = bytes(out)
        assert big.verify_raw(sets, srb, 4) is True
        bad = bytearray(sets)
        bad[9999 * 320 + 100] ^= 0x04
        got = big.verify_raw(bytes(bad), srb, 4, want_gt=True)
        assert got[0] is False
        assert got == br.batch_verify(bytes(bad), srb, 4)
        # the serial derivation (one chain of 16 400) takes the same route
        assert big.verify_raw(bytes(bad), srb, 0, want_gt=True) == br.batch_verify(bytes(bad), srb, 0)
    finally:
        big.close()


def test_device_generated_sets_equal_blst_recipe(cache, br):
    """The benchmark workload generator (k_make_sets: the device's own hash_to_G2 and scalar multiplications) against
    the same recipe computed with BLST on the host (oracle ref_make_sets_device_recipe): byte-identical sets, so the
    batches bench.py times are the ones the reference arm verifies."""
    import nim_blscurve_b200 as bg
    n = 300
    out = (C.c_uint8 * (320 * n))()
    assert bg.lib().blsgpu_make_sets(cache.handle, 2026, 1000, n, out, 0) == 0
    assert bytes(out) == br.make_sets_device_recipe(2026, 1000, n)


def test_large_batch_properties(cache, br, srb):
    """4096 device-generated sets: verdict true; one corrupted set flips it and the GT equals BLST's;
    verdict and GT are independent of the Miller grouping / share split (checksum-of-products property)."""
    import nim_blscurve_b200 as bg
    n = 4096
    out = (C.c_uint8 * (320 * n))()
    assert bg.lib().blsgpu_make_sets(cache.handle, 99, 0, n, out, 0) == 0
    sets = bytes(out)
    assert cache.verify_raw(sets, srb, 64) is True
    bad = bytearray(sets)
    bad[1234 * 320 + 96] ^= 0x80
    ok, gt = cache.verify_raw(bytes(bad), srb, 64, want_gt=True)
    assert ok is False
    rok, rgt = br.batch_verify(bytes(bad), srb, 64)
    assert (ok, gt) == (rok, rgt)
    be = bg.GpuBackend(cache)
    parts = b""
    for r in range(4):
        first, cnt = bg.shard_range(n, 4, r)
        parts += be.partial(bytes(bad)[first * 320:(first + cnt) * 320], first, n, srb, 64)[0]
    assert be.finalize(parts) == (ok, gt)


def test_epoch_batch_full_size_properties(br, srb):
    """The bench workload at full size (131 072 distinct-message sets, the per-GPU share of BASELINE configs[4]) through
    size-independent properties: the valid batch verifies; one flipped message bit anywhere rejects it; the
    post-final-exponentiation GT of the rejected batch does not depend on how the batch is cut into rank shares
    (8 shares cut by the reference chunk rule vs one context); and a 1 500-set window around the corrupted
    set is pinned against BLST."""
    import nim_blscurve_b200 as bg
    n = 131072
    big = bg.BatchedBLSVerifierCache(max_sets=n, device=0)
    try:
        out = (C.c_uint8 * (320 * n))()
        assert bg.lib().blsgpu_make_sets(big.handle, 2026, 0, n, out, 0) == 0
        sets = bytes(out)
        assert big.verify_raw(sets, srb, 1024) is True
        victim = 100003
        bad = bytearray(sets)
        bad[victim * 320 + 96 + 31] ^= 0x01
        bad = bytes(bad)
        ok, gt = big.verify_raw(bad, srb, 1024, want_gt=True)
        assert ok is False
        be = bg.GpuBackend(big)
        parts = b""
        for r in range(8):
            first, cnt = bg.shard_range(n, 8, r)
            parts += be.partial(bad[first * 320:(first + cnt) * 320], first, n, srb, 1024)[0]
        assert be.finalize(parts) == (ok, gt)
        w0 = victim - 700
        window = bad[w0 * 320:(w0 + 1500) * 320]
        assert big.verify_raw(window, srb, 16, want_gt=True) == br.batch_verify(window, srb, 16)
        # the same batch resident in device memory (blsgpu_batch_verify_dev: one launch per stage instead of the sliced
        # copy/hash pipeline of the host call)
        import torch
        L = bg.lib()
        d = torch.frombuffer(bytearray(bad), dtype=torch.uint8).cuda()
        gt2 = (C.c_uint8 * 576)()
        for chunks in (1024, 16):
            rc = L.blsgpu_batch_verify_dev(big.handle, C.c_void_p(d.data_ptr()), n, srb, chunks, None, gt2)
            assert rc == 0, big.last_error()
            if chunks == 1024:
                assert bytes(gt2) == gt
        # a batch just past one wave of blocks (75 776 sets) of the thread-per-set kernels
        n2 = 76000
        rc = L.blsgpu_batch_verify_dev(big.handle, C.c_void_p(d.data_ptr()), n2, srb, 16, None, gt2)
        assert rc == 1, big.last_error()
        rc = L.blsgpu_batch_verify_dev(big.handle, C.c_void_p(d.data_ptr() + 320 * (victim - 75990)), n2, srb, 16, None, gt2)
        assert rc == 0, big.last_error()
        parts = b""
        sub = bad[(victim - 75990) * 320:(victim - 75990 + n2) * 320]
        for r in range(3):
            first, cnt = bg.shard_range(n2, 3, r)
            parts += be.partial(sub[first * 320:(first + cnt) * 320], first, n2, srb, 16)[0]
        assert be.finalize(parts) == (False, bytes(gt2))
    finally:
        big.close()


@pytest.mark.parametrize("n", [127, 128, 129, 1024, 1025, 2047, 2048, 2049, 2499, 2500, 4096, 4097, 4499, 4500, 6000, 8192, 8193, 9000])
def test_route_boundaries_vs_blst(br, srb, n):
    """The batch pipeline picks its kernels by batch size (route.hpp; tests/test_hostsim.py::test_route_plans pins the
    plans): per-set programs up to 4 096 sets, two lanes per message from 2 049, Pippenger for the G2 sum from 2 500,
    the signature pair's own Miller loop from 4 500, graph replay up to 8 192.  One batch on each side of the
    boundaries, valid and with one corrupted set, verdict and GT against BLST."""
    import nim_blscurve_b200 as bg
    c = bg.BatchedBLSVerifierCache(max_sets=n, device=0)
    try:
        out = (C.c_uint8 * (320 * n))()
        assert bg.lib().blsgpu_make_sets(c.handle, 31337, 0, n, out, 0) == 0
        sets = bytes(out)
        assert c.verify_raw(sets, srb, 32) is True
        bad = bytearray(sets)
        bad[(n // 2) * 320 + 100] ^= 0x10         # message of one set (points stay on the curve: inputs are pre-validated)
        assert c.verify_raw(bytes(bad), srb, 32, want_gt=True) == br.batch_verify(bytes(bad), srb, 32)
    finally:
        c.close()


def test_thread_per_set_route_vs_blst(br, srb):
    """The thread-per-set kernels (k_hash_sets, k_miller_lines) serve only very large batches by default (hash beyond
    125 000 sets, lines beyond 180 000 pairs); a child process with the lane-pair routes switched off runs them on a
    9 000-set batch, valid and with one corrupted set, and the verdicts and GT bytes are compared with BLST's here."""
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    code = r'''
import ctypes as C, hashlib, sys
sys.path.insert(0, %r)
import nim_blscurve_b200 as bg
srb = bytes.fromhex(%r)
n = 9000
c = bg.BatchedBLSVerifierCache(max_sets=n, device=0)
out = (C.c_uint8 * (320 * n))()
assert bg.lib().blsgpu_make_sets(c.handle, 4242, 0, n, out, 0) == 0
sets = bytes(out)
print("valid", c.verify_raw(sets, srb, 16))
bad = bytearray(sets); bad[4321 * 320 + 97] ^= 0x02
ok, gt = c.verify_raw(bytes(bad), srb, 16, want_gt=True)
print("bad", ok, gt.hex())
''' % (root, srb.hex())
    env = dict(os.environ, BLSGPU_PAIR_HASH_MAX="1", BLSGPU_PAIR_LINES_MAX="1")
    r = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = r.stdout.strip().splitlines()
    assert lines[0] == "valid True"
    tag, ok, gt_hex = lines[1].split()
    import nim_blscurve_b200 as bg
    c = bg.BatchedBLSVerifierCache(max_sets=9000, device=0)
    try:
        out = (C.c_uint8 * (320 * 9000))()
        assert bg.lib().blsgpu_make_sets(c.handle, 4242, 0, 9000, out, 0) == 0
    finally:
        c.close()
    bad = bytearray(bytes(out))
    bad[4321 * 320 + 97] ^= 0x02
    rok, rgt = br.batch_verify(bytes(bad), srb, 16)
    assert (ok == "True", bytes.fromhex(gt_hex)) == (rok, rgt)
