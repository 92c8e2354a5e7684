"""Stand-in for oracle/blst_ref.py when the BLST build (oracle/_ref) is absent — TEST INFRASTRUCTURE ONLY.

Same functions, same return values.  Every answer is computed by, or stored from, the pure-Python restatement
oracle/pyref.py, which tests/test_oracle_golden.py pins to BLST's own outputs; the library under test answers nothing:

* exact group operations (aggregate, subtract, negate, compress, serialize), the decoders (fromBytes with BLST's
  error codes), rank partials and their final exponentiation, and the RLC scalars are computed by pyref at call time;
* inputs (signature sets, MSM points) follow the recipes of oracle/ref_batch.c byte for byte: the IETF KeyGen of
  blst_keygen and the splitmix scalars are computed here, and the scalar multiplications and hash_to_G2 of the
  inputs by the library (INPUTS_ON_DEVICE; pyref when False, which is slow).  A wrong library result makes different
  input bytes, and then no stored answer matches them;
* batch verdicts and GT bytes, MSM results, hash_to_G2 points, combine and aggregate-verify results, too slow for
  pyref at the tests' sizes, are read from tests/golden/oracle_answers.json.gz, keyed by a hash of the call's
  arguments.  tests/test_oracle_golden.py recomputes a sample of every kind of entry with pyref.  With
  BLSGPU_ORACLE_RECORD=<path> missing answers are computed with pyref and the table is written to <path> at exit.

Nothing under ``nim_blscurve_b200/`` may import this module.
"""
import atexit
import base64
import gzip
import hashlib
import hmac
import json
import os

from oracle import pyref as pr

_TABLE = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden",
                      "oracle_answers.json.gz")
_RECORD = os.environ.get("BLSGPU_ORACLE_RECORD")
DST_ETH2 = pr.DST_ETH2
INPUTS_ON_DEVICE = True
_answers = None
_cache = None


def _gpu():
    global _cache
    if _cache is None:
        import nim_blscurve_b200 as bg
        _cache = bg.BatchedBLSVerifierCache(max_sets=64, device=0)
    return _cache


def _enc(v):
    if isinstance(v, (bytes, bytearray)):
        return "b" + base64.b64encode(bytes(v)).decode()
    if isinstance(v, (tuple, list)):
        return [_enc(x) for x in v]
    return v


def _dec(v):
    if isinstance(v, str):
        return base64.b64decode(v[1:])
    if isinstance(v, list):
        return tuple(_dec(x) for x in v)
    return v


def _key(name, args):
    h = hashlib.sha256(name.encode())
    for a in args:
        if isinstance(a, (bytes, bytearray)):
            h.update(b"|b%d:" % len(a) + hashlib.sha256(a).digest())
        elif isinstance(a, (list, tuple)) and all(isinstance(x, (bytes, bytearray)) for x in a):
            h.update(b"|l%d:" % len(a) + hashlib.sha256(b"".join(hashlib.sha256(x).digest() for x in a)).digest())
        else:
            h.update(b"|" + repr(a).encode())
    return h.hexdigest()[:32]


def _write():
    with gzip.open(_RECORD, "wt") as f:
        json.dump(_answers, f, sort_keys=True, separators=(",", ":"))


def _answer(name, args, compute):
    global _answers
    if _answers is None:
        _answers = {}
        if os.path.exists(_TABLE):
            with gzip.open(_TABLE, "rt") as f:
                _answers = json.load(f)
        if _RECORD:
            atexit.register(_write)
    k = _key(name, args)
    if k not in _answers:
        if not _RECORD:
            raise LookupError(f"no stored answer for {name} on these inputs (tests/golden/oracle_answers.json.gz); "
                              "build oracle/_ref to compare with BLST directly")
        _answers[k] = _enc(compute())
    return _dec(_answers[k])


# ---- inputs (oracle/ref_batch.c recipes) -------------------------------------------------------------------------
def keygen(seed):
    """blst_keygen(IKM = LE64(seed) || 0^24, no info): the IETF KeyGen (HKDF-SHA-256, salt re-hashed until sk != 0)."""
    ikm = seed.to_bytes(8, "little") + bytes(24)
    salt, sk = b"BLS-SIG-KEYGEN-SALT-", 0
    while sk == 0:
        salt = hashlib.sha256(salt).digest()
        prk = hmac.new(salt, ikm + b"\x00", hashlib.sha256).digest()
        okm, t = b"", b""
        for i in (1, 2):
            t = hmac.new(prk, t + (48).to_bytes(2, "big") + bytes([i]), hashlib.sha256).digest()
            okm += t
        sk = int.from_bytes(okm[:48], "big") % pr.R_ORDER
    return sk


def _g1_mul_gen(sks):
    if not INPUTS_ON_DEVICE:
        return [pr.g1_to_mem(pr.g1_mul(pr.G1_GEN, k)) for k in sks]
    import nim_blscurve_b200 as bg
    gen = pr.g1_to_mem(pr.G1_GEN)
    return [bg.msmG1(_gpu(), gen, k.to_bytes(32, "little"), 255) for k in sks]


def _hash_g2(msgs, msg_len, dst):
    """Affine H(m) of each message, 192 bytes each."""
    if not INPUTS_ON_DEVICE:
        n = len(msgs) // msg_len if msg_len else 1
        return b"".join(pr.g2_to_mem(pr.hash_to_g2(msgs[msg_len * i:msg_len * (i + 1)], dst)) for i in range(n))
    import nim_blscurve_b200 as bg
    return bg.hashToG2(_gpu(), msgs, msg_len, dst)[1]


def _g2_mul(points192, sks):
    if not INPUTS_ON_DEVICE:
        return [pr.g2_to_mem(pr.g2_mul(pr.g2_from_mem(points192[192 * i:192 * i + 192]), k)) for i, k in enumerate(sks)]
    import nim_blscurve_b200 as bg
    return [bg.msmG2(_gpu(), points192[192 * i:192 * i + 192], k.to_bytes(32, "little"), 255) for i, k in enumerate(sks)]


def _sign_hashed_many(sks, hashed, dst=DST_ETH2):
    """(pk, sig) per key over the 32-byte messages `hashed` (one per key)."""
    return _g1_mul_gen(sks), _g2_mul(_hash_g2(b"".join(hashed), 32, dst), sks)


def make_sets(start_seed, n, msg_prefix=b"msg", threads=0):
    seeds = range(start_seed, start_seed + n)
    hashed = [hashlib.sha256(msg_prefix[:64] + b"%d" % s).digest() for s in seeds]
    pks, sigs = _sign_hashed_many([keygen(s) for s in seeds], hashed) if n else ([], [])
    return b"".join(p + m + s for p, m, s in zip(pks, hashed, sigs))


def make_set(seed, message):
    return sign_hashed(seed, hashlib.sha256(message).digest())


def sign_hashed(seed, hashed32):
    pks, sigs = _sign_hashed_many([keygen(seed)], [hashed32])
    return pks[0] + hashed32 + sigs[0]


def sign(seed, msg, dst=DST_ETH2):
    sk = keygen(seed)
    return _g1_mul_gen([sk])[0], _g2_mul(_hash_g2(msg, len(msg), dst), [sk])[0]


def fast_aggregate_set(start_seed, nkeys, hashed32, threads=0):
    """Member public keys, and the set (sum of keys, message, sum of signatures): the signature sum is [sum sk]H(m)."""
    sks = [keygen(start_seed + i) for i in range(nkeys)]
    pks = _g1_mul_gen(sks)
    sig = _g2_mul(_hash_g2(hashed32, 32, DST_ETH2), [sum(sks) % pr.R_ORDER])[0]
    return b"".join(pks), aggregate_g1(b"".join(pks))[1] + hashed32 + sig


def make_sets_device_recipe(seed, first, n, threads=0):
    """The blsgpu_make_sets recipe (oracle/ref_batch.c ref_make_sets_device_recipe) computed in pure Python."""
    out = b""
    for i in range(first, first + n):
        dig = hashlib.sha256(seed.to_bytes(8, "little") + bytes(24) + i.to_bytes(8, "little")).digest()
        sk = (int.from_bytes(dig, "big") % (1 << 250)) | 1
        msg = hashlib.sha256(b"blsgpu" + i.to_bytes(8, "little")).digest()
        out += pr.g1_to_mem(pr.g1_mul(pr.G1_GEN, sk)) + msg + pr.g2_to_mem(pr.g2_mul(pr.hash_to_g2(msg), sk))
    return out


def _splitmix(s):
    s = (s + 0x9e3779b97f4a7c15) & 0xFFFFFFFFFFFFFFFF
    z = s
    z = ((z ^ (z >> 30)) * 0xbf58476d1ce4e5b9) & 0xFFFFFFFFFFFFFFFF
    z = ((z ^ (z >> 27)) * 0x94d049bb133111eb) & 0xFFFFFFFFFFFFFFFF
    return s, z ^ (z >> 31)


def msm_points(seed, n, threads=0):
    """(points n*96, scalars n*32): point i = [k_i]G1 for a 96-bit k_i, 255-bit scalars (ref_msm_inputs)."""
    ks, sc = [], b""
    for i in range(n):
        s = seed ^ ((0xFACADE + i * 0x100000001b3) & 0xFFFFFFFFFFFFFFFF)
        s, a = _splitmix(s)
        s, b = _splitmix(s)
        ks.append(a | (b & 0xFFFFFFFF) << 64)
        words = []
        for _ in range(4):
            s, v = _splitmix(s)
            words.append(v)
        w = b"".join(v.to_bytes(8, "little") for v in words)
        sc += w[:31] + bytes([w[31] & 0x7f])
    return b"".join(_g1_mul_gen(ks)), sc


# ---- exact group operations (pyref) -------------------------------------------------------------------------------
def rlc_scalars(srb, n, chunks):
    return pr.rlc_scalars(srb, n, chunks)


def _sum(points, size):
    frm, add = (pr.g1_from_mem, pr.g1_add) if size == 96 else (pr.g2_from_mem, pr.g2_add)
    acc = None
    for i in range(0, len(points), size):
        acc = add(acc, frm(points[i:i + size]))
    return acc


def aggregate_g1(points96):
    return (len(points96) > 0, pr.g1_to_mem(_sum(points96, 96)))


def aggregate_g2(points192):
    return (len(points192) > 0, pr.g2_to_mem(_sum(points192, 192)))


def subtract_all(dst, points):
    sz = len(dst)
    assert sz in (96, 192) and len(points) % sz == 0
    if not points:
        return bytes(dst)
    if sz == 96:
        return pr.g1_to_mem(pr.g1_add(pr.g1_from_mem(dst), pr.g1_neg(_sum(points, 96))))
    return pr.g2_to_mem(pr.g2_add(pr.g2_from_mem(dst), pr.g2_neg(_sum(points, 192))))


def g2_neg(aff192):
    return pr.g2_to_mem(pr.g2_neg(pr.g2_from_mem(aff192)))


def g1_compress(aff96):
    return pr.g1_compress(pr.g1_from_mem(aff96))


def g2_compress(aff192):
    return pr.g2_compress(pr.g2_from_mem(aff192))


def g1_serialize(aff96):
    return pr.g1_serialize(pr.g1_from_mem(aff96))


def g2_serialize(aff192):
    return pr.g2_serialize(pr.g2_from_mem(aff192))


# ---- pyref at call time ------------------------------------------------------------------------------------------
def pubkey_from_bytes(raw, group_check=True):
    return pr.pubkey_from_bytes(raw, group_check)


def signature_from_bytes(raw, group_check=True):
    return pr.signature_from_bytes(raw, group_check)


def _sets(raw):
    return [(pr.g1_from_mem(raw[i:i + 96]), raw[i + 96:i + 128], pr.g2_from_mem(raw[i + 128:i + 320]))
            for i in range(0, len(raw), 320)]


def _f12_from_mem(b):
    """BLST's in-memory fp12 (c0, c1 of Fp6, each of three Fp2, Montgomery little-endian limbs)."""
    c = [pr.fp_from_mont_bytes(b[48 * k:48 * k + 48]) for k in range(12)]
    f2 = [(c[2 * k], c[2 * k + 1]) for k in range(6)]
    return ((f2[0], f2[1], f2[2]), (f2[3], f2[4], f2[5]))


def _f12_to_mem(a):
    return b"".join(pr.fp_to_mont_bytes(x) for j in range(2) for i in range(3) for x in a[j][i])


def partial(sets, first, total_n, srb, chunks):
    """One rank's share: conj(ML(S_k, G1)) * prod ML([r_i]pk_i, H(m_i)) with the global scalars, and the flag.  pyref's
    Miller loop differs from BLST's by factors the final exponentiation removes, so only finalize() of a product of
    partials is comparable bit for bit (which is how the tests use it)."""
    n = len(sets) // 320
    if n == 0:
        return _f12_to_mem(pr.F12_ONE), 0
    r = pr.rlc_scalars(srb, total_n, chunks)[first:first + n]
    gt, S = pr.F12_ONE, None
    for (pk, msg, sig), k in zip(_sets(sets), r):
        if pk is None:
            return _f12_to_mem(pr.F12_ONE), 1
        if sig is not None:
            S = pr.g2_add(S, pr.g2_mul(sig, k))
        gt = pr.f12_mul(gt, pr.miller_loop(pr.g1_mul(pk, k), pr.hash_to_g2(msg)))
    gs = pr.miller_loop(pr.G1_GEN, S) if S is not None else pr.F12_ONE
    return _f12_to_mem(pr.f12_mul(pr.f12_conj(gs), gt)), 0


def finalize(partials):
    if not partials:
        return False, bytes(576)
    acc = pr.F12_ONE
    for i in range(0, len(partials), 576):
        acc = pr.f12_mul(acc, _f12_from_mem(partials[i:i + 576]))
    out = pr.final_exp(acc)
    return out == pr.F12_ONE, pr.f12_to_bytes(out)


# ---- stored answers, recorded with pyref --------------------------------------------------------------------------
def _ref_batch_verify(sets, srb, chunks, scalars):
    if not sets:
        return False, bytes(576)
    ok, gt = pr.batch_verify(_sets(sets), srb, chunks, scalars)
    return ok, gt if gt is not None else bytes(576)


def _ref_msm(points, scalars, nbits, g2):
    size = 192 if g2 else 96
    n, sb = len(points) // size, (nbits + 7) // 8
    frm, mul, add, to = (pr.g2_from_mem, pr.g2_mul, pr.g2_add, pr.g2_to_mem) if g2 else \
        (pr.g1_from_mem, pr.g1_mul, pr.g1_add, pr.g1_to_mem)
    acc = None
    for i in range(n):
        k = int.from_bytes(scalars[sb * i:sb * i + sb], "little") & ((1 << nbits) - 1)
        acc = add(acc, mul(frm(points[size * i:size * i + size]), k))
    return to(acc)


def _ref_hash_to_g2(msgs, msg_len, dst):
    n = len(msgs) // msg_len if msg_len else 0
    pts = [pr.hash_to_g2(msgs[msg_len * i:msg_len * (i + 1)], dst) for i in range(n)]
    return b"".join(pr.g2_compress(q) for q in pts), b"".join(pr.g2_to_mem(q) for q in pts)


def _ref_combine(srb, pks, sigs):
    """MultiSignatureSet.combine (blst_min_pubkey_sig_core.nim:570-647, oracle/ref_batch.c ref_combine)."""
    n = len(pks) // 96
    if n == 1:
        return pks, sigs
    seed, avail, sc = srb, 0, []
    while len(sc) < n:
        if avail == 0:
            seed, avail = hashlib.sha256(seed).digest(), 4
        avail -= 1
        v = int.from_bytes(seed[8 * avail:8 * avail + 8], "little")
        if v:
            sc.append(v)
    scb = b"".join(v.to_bytes(8, "little") for v in sc)
    return _ref_msm(pks, scb, 64, False), _ref_msm(sigs, scb, 64, True)


def _ref_aggregate_verify(pks, msgs, sig, dst):
    n = len(pks) // 96
    if n == 0:
        return False, bytes(576)
    gt = pr.F12_ONE
    for i, m in enumerate(msgs):
        pk = pr.g1_from_mem(pks[96 * i:96 * i + 96])
        if pk is None:
            return False, bytes(576)
        gt = pr.f12_mul(gt, pr.miller_loop(pk, pr.hash_to_g2(m, dst)))
    s = pr.g2_from_mem(sig)
    gs = pr.miller_loop(pr.G1_GEN, s) if s is not None else pr.F12_ONE
    out = pr.final_exp(pr.f12_mul(pr.f12_conj(gs), gt))
    return out == pr.F12_ONE, pr.f12_to_bytes(out)


def _ref_fast_aggregate_verify(pks, msg, sig, dst):
    ok, agg = aggregate_g1(pks)
    if not ok:
        return False, bytes(576)
    return _ref_aggregate_verify(agg, [msg], sig, dst)


def batch_verify(sets, srb, chunks=0, scalars=None):
    return _answer("batch_verify", (sets, srb, chunks, scalars), lambda: _ref_batch_verify(sets, srb, chunks, scalars))


def msm_g1(points96, scalars32, nbits=255):
    return _answer("msm_g1", (points96, scalars32, nbits), lambda: _ref_msm(points96, scalars32, nbits, False))


def msm_g2(points192, scalars, nbits=255):
    return _answer("msm_g2", (points192, scalars, nbits), lambda: _ref_msm(points192, scalars, nbits, True))


def hash_to_g2(msgs, msg_len, dst):
    return _answer("hash_to_g2", (msgs, msg_len, dst), lambda: _ref_hash_to_g2(msgs, msg_len, dst))


def combine(srb, pubkeys96, sigs192):
    return _answer("combine", (srb, pubkeys96, sigs192), lambda: _ref_combine(srb, pubkeys96, sigs192))


def aggregate_verify(pubkeys96, msgs, sig192, dst=DST_ETH2):
    return _answer("aggregate_verify", (pubkeys96, list(msgs), sig192, dst),
                   lambda: _ref_aggregate_verify(pubkeys96, list(msgs), sig192, dst))


def fast_aggregate_verify(pubkeys96, msg, sig192, dst=DST_ETH2):
    return _answer("fast_aggregate_verify", (pubkeys96, msg, sig192, dst),
                   lambda: _ref_fast_aggregate_verify(pubkeys96, msg, sig192, dst))
