"""GPU parity: batch verification through the C ABI vs BLST (oracle/_ref) on the scenarios of
/root/reference/tests/t_batch_verifier.nim — verify boolean AND the 576-byte GT must match."""
import hashlib
import random

import pytest

pytestmark = pytest.mark.gpu


def both(cache, br, sets, srb, chunks, scalars=None):
    ok, gt = cache.verify_raw(sets, srb, chunks, scalars=scalars, want_gt=True)
    rok, rgt = br.batch_verify(sets, srb, chunks, scalars=scalars)
    assert ok == rok
    assert gt == rgt
    return ok


def examples(br, n):
    # addExample(i, "msg" & $i)  (t_batch_verifier.nim:42-47)
    return br.make_sets(0, n, b"msg")


@pytest.mark.parametrize("n", [1, 2, 15, 16, 17])
@pytest.mark.parametrize("chunks", [0, 4])
def test_valid_batches(cache, br, srb, n, chunks):
    assert both(cache, br, examples(br, n), srb, chunks) is True


@pytest.mark.parametrize("chunks", [0, 4])
def test_config0_64_sets(cache, br, srb, chunks):
    """BASELINE configs[0] exactly: 64 distinct-message sets (SURVEY.md section 8d config 1: sk_i from ikm LE64(i),
    m_i = SHA256("msg" || dec(i)), srb = SHA256("Mr F was here")), serial and 4-chunk derivations, plus the two negative
    variants of tests/t_batch_verifier.nim at that size: one wrong signature (:122-137) and one forged pair (:198-244)."""
    sets = examples(br, 64)
    assert both(cache, br, sets, srb, chunks) is True
    wrong = bytearray(sets)
    wrong[17 * 320 + 128:18 * 320] = sets[40 * 320 + 128:41 * 320]      # (pubkey17, msg17, sig40)
    assert both(cache, br, bytes(wrong), srb, chunks) is False
    forged = sets[:62 * 320] + forged_pair(br, cache, 3, b"msg300", 4, b"msg400")
    assert len(forged) == 64 * 320
    assert both(cache, br, forged, srb, chunks) is False


@pytest.mark.parametrize("chunks", [0, 4])
def test_wrong_signature(cache, br, srb, chunks):
    s1 = br.make_set(1, b"msg1")
    s2 = br.make_set(2, b"msg2")
    bad = s1 + s2[:128] + s1[128:]          # (pubkey2, msg2, sig1)   t_batch_verifier.nim:122-137
    assert both(cache, br, bad, srb, chunks) is False


def forged_pair(br, cache, seed1, m1, seed2, m2):
    """S1+S', S2-S' (t_batch_verifier.nim:198-244)."""
    import nim_blscurve_b200 as bg
    a, b = br.make_set(seed1, m1), br.make_set(seed2, m2)
    p = br.make_set(seed1 * seed2 + seed1 + seed2, b"rekt")
    sp = p[128:]
    nsp = br.g2_neg(sp)
    ok1, f1 = br.aggregate_g2(a[128:] + sp)
    ok2, f2 = br.aggregate_g2(b[128:] + nsp)
    assert ok1 and ok2
    # the same aggregation on the GPU must give the same points
    g1 = bg.aggregateAll(cache, [a[128:], sp])
    g2 = bg.aggregateAll(cache, [b[128:], nsp])
    assert g1 == (True, f1) and g2 == (True, f2)
    return a[:128] + f1 + b[:128] + f2


@pytest.mark.parametrize("chunks", [0, 4])
def test_forged_pair(cache, br, srb, chunks):
    batch = forged_pair(br, cache, 1, b"msg1", 2, b"msg2")
    assert both(cache, br, batch, srb, chunks) is False


@pytest.mark.parametrize("chunks", [0, 4])
def test_one_forgery_among_many(cache, br, srb, chunks):
    sets = examples(br, 16) + forged_pair(br, cache, 1, b"msg100", 2, b"msg200")
    items = [sets[i:i + 320] for i in range(0, len(sets), 320)]
    random.Random(1234).shuffle(items)
    assert both(cache, br, b"".join(items), srb, chunks) is False


def test_same_message_100(cache, br, srb):
    msg = hashlib.sha256(b"msg").digest()
    sets = b"".join(br.sign_hashed(i, msg) for i in range(100))
    assert both(cache, br, sets, srb, 4) is True


def test_empty_is_false(cache, srb):
    assert cache.verify_raw(b"", srb, 0) is False
    import nim_blscurve_b200 as bg
    assert bg.batchVerify(bg.Taskpool.new(4), cache, [], srb) is False


def test_infinite_pubkey_fails(cache, br, srb):
    sets = bytearray(examples(br, 5))
    sets[2 * 320:2 * 320 + 96] = bytes(96)
    sets[2 * 320 + 128:3 * 320] = bytes(192)        # infinite pk AND infinite sig still fails (aggregate.c:296)
    ok, gt = cache.verify_raw(bytes(sets), srb, 0, want_gt=True)
    rok, _ = br.batch_verify(bytes(sets), srb, 0)
    assert ok is False and rok is False


def test_infinite_signature_is_skipped(cache, br, srb):
    sets = bytearray(examples(br, 4))
    sets[320 + 128:640] = bytes(192)
    assert both(cache, br, bytes(sets), srb, 0) is False
    # all signatures infinite: GTsig := one (aggregate.c:486-492)
    for i in range(4):
        sets[i * 320 + 128:(i + 1) * 320] = bytes(192)
    assert both(cache, br, bytes(sets), srb, 4) is False


def test_explicit_scalars(cache, br, srb):
    sets = examples(br, 9)
    sc = [random.Random(7).getrandbits(64) | 1 for _ in range(9)]
    assert both(cache, br, sets, srb, 0, scalars=sc) is True
    bad = bytearray(sets)
    bad[128:320] = sets[320 + 128:640]
    assert both(cache, br, bytes(bad), srb, 0, scalars=sc) is False


def test_api_mirror(cache, br, srb):
    import nim_blscurve_b200 as bg
    tp = bg.Taskpool.new(numThreads=4)
    raw = examples(br, 6)
    batch = [bg.SignatureSet(raw[i:i + 96], raw[i + 96:i + 128], raw[i + 128:i + 320]) for i in range(0, len(raw), 320)]
    assert bg.batchVerify(tp, cache, batch, srb)
    assert bg.batchVerifySerial(cache, batch, srb)
    assert bg.batchVerifyParallel(tp, cache, batch, srb)
    assert bg.batchVerify(tp, cache, batch[:2], srb)       # < 3 sets -> serial path


@pytest.mark.parametrize("n,chunks", [(10, 0), (10, 4), (3, 8), (257, 16), (1000, 7)])
def test_rlc_scalars(cache, srb, n, chunks):
    """Against pyref's restatement of the derivation (pinned to BLST's scalars by tests/test_oracle_golden.py)."""
    import nim_blscurve_b200 as bg
    from oracle import pyref as pr
    assert bg.rlcScalars(cache, srb, n, chunks) == pr.rlc_scalars(srb, n, chunks)


def test_device_generated_sets_verify(cache, br, srb):
    """The benchmark's synthetic generator must produce sets BLST accepts."""
    import ctypes as C
    import nim_blscurve_b200 as bg
    n = 40
    out = (C.c_uint8 * (320 * n))()
    rc = bg.lib().blsgpu_make_sets(cache.handle, 42, 1000, n, out, 0)
    assert rc == 0
    sets = bytes(out)
    assert both(cache, br, sets, srb, 4) is True
    assert len({sets[i + 96:i + 128] for i in range(0, len(sets), 320)}) == n     # distinct messages
    bad = bytearray(sets)
    bad[5 * 320 + 96] ^= 1                                                        # flip one message bit
    assert both(cache, br, bytes(bad), srb, 4) is False


@pytest.mark.parametrize("n", [1, 2, 5, 100, 1000])
def test_combine_same_message(cache, br, srb, n):
    """MultiSignatureSet.combine (tests/t_batch_verifier.nim:159-177): same scalars, same Pippenger results as BLST,
    and the combined set verifies like the reference's."""
    import nim_blscurve_b200 as bg
    sets = [br.make_set(i, b"same message") for i in range(n)]   # (pk, SHA256(text), sig) on one message
    msg = sets[0][96:128]
    pks = [s[:96] for s in sets]
    sigs = [s[128:320] for s in sets]
    pk, sig = bg.combine(cache, srb, pks, sigs)
    assert (pk, sig) == br.combine(srb, b"".join(pks), b"".join(sigs))
    ms = bg.MultiSignatureSet(pks, msg, sigs)
    one = ms.combine(cache, srb)
    assert bg.batchVerifySerial(cache, [one], srb) == br.batch_verify(one.to_bytes(), srb, 0)[0] is True
    # a shuffled signature list must fail (t_batch_verifier.nim:171-177)
    if n >= 2:
        bad = bg.MultiSignatureSet(pks, msg, sigs[1:] + sigs[:1]).combine(cache, srb)
        assert bg.batchVerifySerial(cache, [bad], srb) is False


def test_concurrent_caches_from_host_threads(br, srb):
    """SURVEY §8(b) threading: concurrent callers each own a cache (bls_batch_verifier.nim:389-391).  Four host
    threads, four contexts on one device, different batch sizes (both kernel routes) and a corrupted batch, several
    rounds at once: every call returns the verdict and GT bytes BLST gives for its batch."""
    import threading
    import nim_blscurve_b200 as bg
    jobs = []
    for t, (n, chunks) in enumerate([(5, 0), (129, 4), (700, 16), (4300, 8)]):
        sets = br.make_sets(3000 + 5000 * t, n)
        if t % 2:
            sets = sets[:320 + 128] + sets[128:320] + sets[640:]      # set 1 carries set 0's signature
        jobs.append((sets, chunks, br.batch_verify(sets, srb, chunks)))
    assert [j[2][0] for j in jobs] == [True, False, True, False]
    errors = []
    start = threading.Barrier(len(jobs))

    def worker(sets, chunks, want):
        try:
            c = bg.BatchedBLSVerifierCache(max_sets=len(sets) // 320, device=0)
            start.wait()
            for _ in range(4):
                got = c.verify_raw(sets, srb, chunks, want_gt=True)
                if got != want:
                    errors.append((len(sets) // 320, got[0], want[0]))
            c.close()
        except Exception as e:      # noqa: BLE001
            errors.append(repr(e))
            start.abort()

    th = [threading.Thread(target=worker, args=j) for j in jobs]
    for x in th:
        x.start()
    for x in th:
        x.join()
    assert errors == []


def test_contexts_on_two_devices_in_one_process(br, srb):
    """One host process driving several GPUs (a Nim application holds one cache per device): contexts on devices 0 and 1
    used alternately and then from two threads, small and large route, give BLST's verdict and GT bytes on both."""
    import threading
    import nim_blscurve_b200 as bg
    if bg.lib().blsgpu_device_count() < 2:
        pytest.skip("needs two devices")
    caches = [bg.BatchedBLSVerifierCache(max_sets=4300, device=d) for d in (0, 1)]
    cases = []
    for n, chunks in [(9, 0), (129, 4), (4300, 8)]:
        sets = br.make_sets(900 + n, n)
        cases.append((sets, chunks, br.batch_verify(sets, srb, chunks)))
    for sets, chunks, want in cases:
        for c in caches:
            assert c.verify_raw(sets, srb, chunks, want_gt=True) == want
    errors = []

    def worker(c):
        for sets, chunks, want in cases * 2:
            if c.verify_raw(sets, srb, chunks, want_gt=True) != want:
                errors.append(len(sets) // 320)

    th = [threading.Thread(target=worker, args=(c,)) for c in caches]
    for x in th:
        x.start()
    for x in th:
        x.join()
    for c in caches:
        c.close()
    assert errors == []


def test_error_convention_of_the_c_abi(br, srb):
    """SURVEY §8(b) error convention: argument / capacity problems are distinct negative codes with a message, never a
    verdict, and a context keeps working after one (the reference doAsserts on an undersized cache,
    bls_batch_verifier.nim:141, :319)."""
    import ctypes as C
    import nim_blscurve_b200 as bg
    L = bg.lib()
    ERR_ARG, ERR_CAPACITY = -2, -3                                   # include/blsgpu.h
    assert L.blsgpu_create(10 ** 6, 16) is None
    assert b"bad device" in L.blsgpu_last_error(None)
    h = L.blsgpu_create(0, 16)
    assert h and L.blsgpu_capacity(h) == 16
    sets = br.make_sets(40, 17)
    gt = (C.c_uint8 * 576)()
    assert L.blsgpu_batch_verify(h, sets, 17, srb, 0, None, gt) == ERR_CAPACITY
    assert b"capacity" in L.blsgpu_last_error(h)
    assert L.blsgpu_batch_verify(h, None, 4, srb, 0, None, gt) == ERR_ARG
    assert L.blsgpu_batch_verify(h, sets, 4, None, 0, None, gt) == ERR_ARG
    assert L.blsgpu_batch_verify(h, sets, 4, srb, 0, (C.c_uint64 * 4)(1, 2, 0, 4), gt) == ERR_ARG      # zero scalar
    assert L.blsgpu_batch_verify(None, sets, 4, srb, 0, None, gt) == ERR_ARG
    assert L.blsgpu_batch_verify(h, sets, 0, srb, 0, None, gt) == 0                                   # empty -> false (:137-139)
    assert L.blsgpu_rlc_scalars(h, srb, 17, 0, (C.c_uint64 * 17)()) == ERR_CAPACITY
    assert L.blsgpu_hash_to_g2(h, b"x", 1, 1, b"d" * 256, 256, None, (C.c_uint8 * 192)()) == ERR_ARG  # DST > 255
    assert L.blsgpu_subtract_g1(h, None, sets[:96], 1) == ERR_ARG
    # the context is still good
    assert L.blsgpu_batch_verify(h, sets, 16, srb, 4, None, gt) == 1
    assert (True, bytes(gt)) == br.batch_verify(sets[:16 * 320], srb, 4)
    L.blsgpu_destroy(h)


def test_graph_replay_follows_the_random_bytes(br):
    """Small batches replay a captured CUDA graph from the third call with the same (buffer, n, chunks) on
    (blsgpu.cu verify_graphed); the 32 random bytes are the one input that changes between replays and reach the scalar
    kernel through device memory.  A failing batch's GT depends on every scalar, so it must follow BLST's for each new
    secureRandomBytes — direct call, capture call and replays alike — and a corrupted copy in the same buffer must be seen."""
    import nim_blscurve_b200 as bg
    c = bg.BatchedBLSVerifierCache(max_sets=64, device=0)
    try:
        sets = bytearray(br.make_sets(0, 33))
        sets[5 * 320 + 128:6 * 320] = sets[6 * 320 + 128:7 * 320]       # wrong signature on set 5
        sets = bytes(sets)
        for k in range(6):
            srb_k = hashlib.sha256(b"replay %d" % k).digest()
            assert c.verify_raw(sets, srb_k, 4, want_gt=True) == br.batch_verify(sets, srb_k, 4), k
        good = br.make_sets(100, 33)
        for k in range(3):
            srb_k = hashlib.sha256(b"valid %d" % k).digest()
            assert c.verify_raw(good, srb_k, 4) is True
            assert c.verify_raw(sets, srb_k, 4) is False
    finally:
        c.close()
