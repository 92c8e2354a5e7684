"""Host-side mirror of blscurve/bls_batch_verifier.nim over the C ABI (include/blsgpu.h).

Names, argument meaning and error behaviour follow the reference:
  * SignatureSet = (pubkey, message, signature)                       bls_batch_verifier.nim:34
    pubkey 96 B / message 32 B / signature 192 B in the reference's in-memory format.
  * BatchedBLSVerifierCache.init() / .init(tp)                          :108-119
  * batchVerifySerial(cache, input, secureRandomBytes)                 :121-160
  * batchVerifyParallel(tp, cache, input, secureRandomBytes)           :296-397
  * batchVerify(tp, cache, input, secureRandomBytes)                   :420-495  (parallel iff
    tp.numThreads > 1 and len >= 3, :440, :468)
  * batchVerifyCompressed(tp, cache, input, secureRandomBytes)         Signature.fromBytes (bls_sig_io.nim:42-60) of
    every SignatureSetCompressed + batchVerify, decoded and subgroup-checked on the device -> (bool, status)
  * aggregateAll(elems) -> (ok, point)                                 blst_min_pubkey_sig_core.nim:179-195
  * subtractAll(dst, elems) -> point                                   blst_min_pubkey_sig_core.nim:197-209
The Taskpool argument stays in the signatures; it no longer fans work out to threads — its
numThreads only selects the reference's RLC-scalar chunking so results are identical for a given tp.
"""
import ctypes as C
from typing import NamedTuple, Optional, Sequence

from ._lib import BlsGpuError, lib


class SignatureSet(NamedTuple):
    pubkey: bytes     # 96 B blst_p1_affine
    message: bytes    # 32 B
    signature: bytes  # 192 B blst_p2_affine

    def to_bytes(self) -> bytes:
        assert len(self.pubkey) == 96 and len(self.message) == 32 and len(self.signature) == 192
        return self.pubkey + self.message + self.signature


class SignatureSetCompressed(NamedTuple):
    """A set as it comes off the network: the signature still in its 96-byte Zcash compressed encoding."""
    pubkey: bytes     # 96 B blst_p1_affine
    message: bytes    # 32 B
    signature: bytes  # 96 B compressed (bls_sig_io.nim:20-36)

    def to_bytes(self) -> bytes:
        assert len(self.pubkey) == 96 and len(self.message) == 32 and len(self.signature) == 96
        return self.pubkey + self.message + self.signature


class Taskpool:
    """Stand-in for taskpools.Taskpool: only numThreads is consulted (scalar chunking)."""

    def __init__(self, numThreads: int = 1):
        self.numThreads = int(numThreads)

    @classmethod
    def new(cls, numThreads: int = 1):
        return cls(numThreads)

    def shutdown(self):
        pass


def _pack(sets) -> bytes:
    if isinstance(sets, (bytes, bytearray, memoryview)):
        b = bytes(sets)
        assert len(b) % 320 == 0
        return b
    return b"".join(s.to_bytes() if isinstance(s, SignatureSet) else SignatureSet(*s).to_bytes() for s in sets)


def _pack_compressed(sets) -> bytes:
    if isinstance(sets, (bytes, bytearray, memoryview)):
        b = bytes(sets)
        assert len(b) % 224 == 0
        return b
    return b"".join(s.to_bytes() if isinstance(s, SignatureSetCompressed) else SignatureSetCompressed(*s).to_bytes()
                    for s in sets)


class BatchedBLSVerifierCache:
    """Device scratch for batch verification (replaces the per-thread pairing contexts, :62-69)."""

    def __init__(self, max_sets: int = 1 << 14, device: int = 0, numThreads: int = 1,
                 devices: Optional[Sequence[int]] = None):
        """devices: several GPUs behind ONE cache (blsgpu_create_multi): batch verification and the MSMs are cut over
        them inside the call, replacing the Taskpools fan-out of bls_batch_verifier.nim:316-369."""
        L = lib()
        if L.blsgpu_device_count() <= 0:
            raise BlsGpuError("no CUDA device visible: nim_blscurve_b200 has no CPU fallback")
        self.devices = list(devices) if devices else None
        if self.devices:
            arr = (C.c_int * len(self.devices))(*self.devices)
            self._h = L.blsgpu_create_multi(arr, len(self.devices), max_sets)
            device = self.devices[0]
        else:
            self._h = L.blsgpu_create(device, max_sets)
        if not self._h:
            raise BlsGpuError(L.blsgpu_last_error(None).decode())
        self.numThreads = numThreads
        self.device = device

    @classmethod
    def init(cls, tp: Optional[Taskpool] = None, max_sets: int = 1 << 14, device: int = 0):
        return cls(max_sets=max_sets, device=device, numThreads=tp.numThreads if tp else 1)

    @property
    def handle(self):
        return self._h

    def capacity(self) -> int:
        return lib().blsgpu_capacity(self._h)

    def last_error(self) -> str:
        return lib().blsgpu_last_error(self._h).decode()

    def close(self):
        if getattr(self, "_h", None):
            lib().blsgpu_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- raw calls -------------------------------------------------------------------------
    def _ensure(self, n):
        if n > self.capacity():
            dev, devs = self.device, self.devices
            self.close()
            self.__init__(max_sets=max(n, 1), device=dev, numThreads=self.numThreads, devices=devs)

    def verify_raw(self, sets: bytes, srb: bytes, chunks: int, scalars: Optional[Sequence[int]] = None,
                   want_gt: bool = False):
        n = len(sets) // 320
        self._ensure(n)
        gt = (C.c_uint8 * 576)() if want_gt else None
        sc = (C.c_uint64 * n)(*scalars) if scalars is not None else None
        rc = lib().blsgpu_batch_verify(self._h, sets, n, srb, chunks, sc, gt)
        if rc < 0:
            raise BlsGpuError(f"blsgpu_batch_verify failed ({rc}): {self.last_error()}")
        return (bool(rc), bytes(gt)) if want_gt else bool(rc)

    def verify_compressed_raw(self, sets: bytes, srb: bytes, chunks: int, scalars: Optional[Sequence[int]] = None,
                              want_gt: bool = False):
        """224-byte compressed sets -> (ok, [BLST_ERROR per set]) or (ok, status, gt)."""
        n = len(sets) // 224
        self._ensure(n)
        gt = (C.c_uint8 * 576)() if want_gt else None
        sc = (C.c_uint64 * n)(*scalars) if scalars is not None else None
        st = (C.c_uint8 * n)()
        rc = lib().blsgpu_batch_verify_compressed(self._h, sets, n, srb, chunks, sc, gt, st)
        if rc < 0:
            raise BlsGpuError(f"blsgpu_batch_verify_compressed failed ({rc}): {self.last_error()}")
        return (bool(rc), list(st), bytes(gt)) if want_gt else (bool(rc), list(st))


def batchVerifyCompressed(tp: Taskpool, cache: BatchedBLSVerifierCache, input, secureRandomBytes: bytes):
    """Signature.fromBytes of every signature (decode + subgroup check, on the device) + batchVerify in one call:
    (verdict, [BLST_ERROR per set]).  A set whose signature fails to decode or is outside G2 fails the batch.  Scalar
    chunking as batchVerify (parallel derivation iff tp.numThreads > 1 and len >= 3); empty input is (False, [])."""
    sets = _pack_compressed(input)
    n = len(sets) // 224
    if n == 0:
        return False, []
    return cache.verify_compressed_raw(sets, secureRandomBytes, max(1, tp.numThreads) if tp.numThreads > 1 and n >= 3 else 0)


def batchVerifySerial(cache: BatchedBLSVerifierCache, input, secureRandomBytes: bytes) -> bool:
    sets = _pack(input)
    if len(sets) == 0:
        return False
    return cache.verify_raw(sets, secureRandomBytes, 0)


def batchVerifyParallel(tp: Taskpool, cache: BatchedBLSVerifierCache, input, secureRandomBytes: bytes) -> bool:
    sets = _pack(input)
    if len(sets) == 0:
        return False
    return cache.verify_raw(sets, secureRandomBytes, max(1, tp.numThreads))


def batchVerify(tp: Taskpool, cache: BatchedBLSVerifierCache, input, secureRandomBytes: bytes) -> bool:
    sets = _pack(input)
    n = len(sets) // 320
    if tp.numThreads > 1 and n >= 3:
        return batchVerifyParallel(tp, cache, sets, secureRandomBytes)
    return batchVerifySerial(cache, sets, secureRandomBytes)


def aggregateAll(cache: BatchedBLSVerifierCache, elems: Sequence[bytes]):
    """Sum of public keys (96 B each) or signatures (192 B each) -> (ok, affine point bytes)."""
    if len(elems) == 0:
        return False, b""
    sz = len(elems[0])
    assert sz in (96, 192) and all(len(e) == sz for e in elems)
    buf = b"".join(elems)
    out = (C.c_uint8 * sz)()
    fn = lib().blsgpu_aggregate_g1 if sz == 96 else lib().blsgpu_aggregate_g2
    rc = fn(cache.handle, buf, len(elems), out)
    if rc < 0:
        raise BlsGpuError(f"aggregate failed ({rc}): {cache.last_error()}")
    return bool(rc), bytes(out)


def subtractAll(cache: BatchedBLSVerifierCache, dst: bytes, elems: Sequence[bytes]) -> bytes:
    """dst - sum(elems) for public keys (96 B) or signatures (192 B); an empty `elems` returns dst unchanged
    (blst_min_pubkey_sig_core.nim:197-209; the Nim proc updates `dst` in place, this mirror returns the new value)."""
    sz = len(dst)
    assert sz in (96, 192) and all(len(e) == sz for e in elems)
    if len(elems) == 0:
        return bytes(dst)
    out = (C.c_uint8 * sz).from_buffer_copy(dst)
    fn = lib().blsgpu_subtract_g1 if sz == 96 else lib().blsgpu_subtract_g2
    rc = fn(cache.handle, out, b"".join(elems), len(elems))
    if rc != 1:
        raise BlsGpuError(f"subtract failed ({rc}): {cache.last_error()}")
    return bytes(out)


def hashToG2(cache: BatchedBLSVerifierCache, msgs: bytes, msg_len: int, dst: bytes):
    """(compressed n*96, affine n*192)"""
    n = len(msgs) // msg_len if msg_len else 1
    comp, aff = (C.c_uint8 * (96 * n))(), (C.c_uint8 * (192 * n))()
    rc = lib().blsgpu_hash_to_g2(cache.handle, msgs if msg_len else None, n, msg_len, dst, len(dst), comp, aff)
    if rc < 0:
        raise BlsGpuError(f"hash_to_g2 failed ({rc}): {cache.last_error()}")
    return bytes(comp), bytes(aff)


def msmG1(cache: BatchedBLSVerifierCache, points96: bytes, scalars: bytes, nbits: int = 255) -> bytes:
    n = len(points96) // 96
    out = (C.c_uint8 * 96)()
    rc = lib().blsgpu_msm_g1(cache.handle, points96, scalars, n, nbits, out)
    if rc < 0:
        raise BlsGpuError(f"msm_g1 failed ({rc}): {cache.last_error()}")
    return bytes(out)


def msmG2(cache: BatchedBLSVerifierCache, points192: bytes, scalars: bytes, nbits: int = 255) -> bytes:
    """sum_i [k_i] Q_i in G2, affine (blst_p2s_mult_pippenger + to_affine; multi_scalar.c:442-446)."""
    n = len(points192) // 192
    out = (C.c_uint8 * 192)()
    rc = lib().blsgpu_msm_g2(cache.handle, points192, scalars, n, nbits, out)
    if rc < 0:
        raise BlsGpuError(f"msm_g2 failed ({rc}): {cache.last_error()}")
    return bytes(out)


class MultiSignatureSet:
    """Signatures that all pertain to the same message (bls_batch_verifier.nim:47-62, init :73-91, add :93-98)."""

    def __init__(self, pubkeys: Sequence[bytes], message: bytes, signatures: Sequence[bytes]):
        assert len(pubkeys) == len(signatures) and len(pubkeys) > 0
        self.pubkeys, self.message, self.signatures = list(pubkeys), message, list(signatures)

    @classmethod
    def init(cls, *args):
        if len(args) == 1:                                   # init(T, sigset)
            ss = args[0] if isinstance(args[0], SignatureSet) else SignatureSet(*args[0])
            return cls([ss.pubkey], ss.message, [ss.signature])
        return cls(*args)

    def add(self, sigset):
        ss = sigset if isinstance(sigset, SignatureSet) else SignatureSet(*sigset)
        assert ss.message == self.message
        self.pubkeys.append(ss.pubkey)
        self.signatures.append(ss.signature)

    def combine(self, cache: "BatchedBLSVerifierCache", secureRandomBytes: bytes) -> SignatureSet:
        """bls_batch_verifier.nim:100-106: one SignatureSet = random linear combination of the members."""
        pk, sig = combine(cache, secureRandomBytes, self.pubkeys, self.signatures)
        return SignatureSet(pk, self.message, sig)


def combine(cache: BatchedBLSVerifierCache, secureRandomBytes: bytes, publicKeys: Sequence[bytes],
            signatures: Sequence[bytes]):
    """blst_min_pubkey_sig_core.nim:570-647 on the device: (sum r_i pk_i, sum r_i sig_i), both affine."""
    assert len(publicKeys) == len(signatures)
    n = len(publicKeys)
    if n == 0:
        raise AssertionError("Must provide at least 1 signature")
    pk, sig = (C.c_uint8 * 96)(), (C.c_uint8 * 192)()
    rc = lib().blsgpu_combine(cache.handle, secureRandomBytes, b"".join(publicKeys), b"".join(signatures), n, pk, sig)
    if rc < 0:
        raise BlsGpuError(f"combine failed ({rc}): {cache.last_error()}")
    return bytes(pk), bytes(sig)


def rlcScalars(cache: BatchedBLSVerifierCache, srb: bytes, n: int, chunks: int):
    out = (C.c_uint64 * n)()
    rc = lib().blsgpu_rlc_scalars(cache.handle, srb, n, chunks, out)
    if rc < 0:
        raise BlsGpuError(f"rlc_scalars failed ({rc}): {cache.last_error()}")
    return list(out)


# ---- blscurve/bls_sig_min_pubkey.nim: aggregateVerify :155-204, fastAggregateVerify :238-258, verify :108-125 ----
DST = b"BLS_SIG_BLS12381G2_XMD:SHA-256_SSWU_RO_POP_"          # bls_sig_min_pubkey.nim:31


def _check(rc, what, cache):
    if rc < 0:
        raise BlsGpuError(f"{what} failed ({rc}): {cache.last_error()}")
    return bool(rc)


def aggregateVerify(cache: BatchedBLSVerifierCache, publicKeys: Sequence[bytes], messages: Sequence[bytes],
                    signature: bytes, dst: bytes = DST, want_gt: bool = False):
    """One signature over n (public key, message) pairs; False on length mismatch or n == 0 (:164-169)."""
    if len(publicKeys) != len(messages) or len(publicKeys) < 1:
        return (False, bytes(576)) if want_gt else False
    offs, o = [0], 0
    for m in messages:
        o += len(m)
        offs.append(o)
    gt = (C.c_uint8 * 576)()
    rc = lib().blsgpu_aggregate_verify(cache.handle, b"".join(publicKeys), len(publicKeys), b"".join(messages) or None,
                                       (C.c_uint32 * len(offs))(*offs), dst, len(dst), signature, gt)
    ok = _check(rc, "aggregate_verify", cache)
    return (ok, bytes(gt)) if want_gt else ok


def verify(cache: BatchedBLSVerifierCache, publicKey: bytes, message: bytes, signature: bytes, dst: bytes = DST) -> bool:
    """coreVerifyNoGroupCheck (blst_min_pubkey_sig_core.nim:264-297) = the one-pair case."""
    return aggregateVerify(cache, [publicKey], [message], signature, dst)


def fastAggregateVerify(cache: BatchedBLSVerifierCache, publicKeys: Sequence[bytes], message: bytes, signature: bytes,
                        dst: bytes = DST, want_gt: bool = False):
    """aggregateAll(publicKeys) on the device, then verify; False on an empty key list (:251-253)."""
    if len(publicKeys) == 0:
        return (False, bytes(576)) if want_gt else False
    gt = (C.c_uint8 * 576)()
    rc = lib().blsgpu_fast_aggregate_verify(cache.handle, b"".join(publicKeys), len(publicKeys), message or None,
                                            len(message), dst, len(dst), signature, gt)
    ok = _check(rc, "fast_aggregate_verify", cache)
    return (ok, bytes(gt)) if want_gt else ok


def aggregateAllSegments(cache: BatchedBLSVerifierCache, groups: Sequence[Sequence[bytes]]):
    """aggregateAll for many committees in one launch -> [(ok, 96-byte point)], ok False for an empty committee."""
    offs, o, flat = [0], 0, []
    for g in groups:
        o += len(g)
        offs.append(o)
        flat.extend(g)
    if not groups:
        return []
    out = (C.c_uint8 * (96 * len(groups)))()
    rc = lib().blsgpu_aggregate_g1_segments(cache.handle, b"".join(flat) or None, (C.c_uint32 * len(offs))(*offs),
                                            len(groups), out)
    _check(rc, "aggregate_g1_segments", cache)
    raw = bytes(out)
    return [(len(g) > 0, raw[96 * i:96 * i + 96]) for i, g in enumerate(groups)]


# ---- blscurve/blst/bls_sig_io.nim:42-122: fromBytes / fromBytesKnownOnCurve, batched ----
def publicKeysFromBytes(cache: BatchedBLSVerifierCache, raw: bytes, size: int = 48, group_check: bool = True):
    """n encodings of `size` (48 or 96) bytes -> (points n*96, [BLST_ERROR per element]); element ok iff status 0."""
    n = len(raw) // size
    out, st = (C.c_uint8 * (96 * n))(), (C.c_uint8 * n)()
    _check(lib().blsgpu_pubkeys_from_bytes(cache.handle, raw, n, size, 1 if group_check else 0, out, st),
           "pubkeys_from_bytes", cache)
    return bytes(out), list(st)


def signaturesFromBytes(cache: BatchedBLSVerifierCache, raw: bytes, size: int = 96, group_check: bool = True):
    n = len(raw) // size
    out, st = (C.c_uint8 * (192 * n))(), (C.c_uint8 * n)()
    _check(lib().blsgpu_signatures_from_bytes(cache.handle, raw, n, size, 1 if group_check else 0, out, st),
           "signatures_from_bytes", cache)
    return bytes(out), list(st)


def publicKeysToBytes(cache: BatchedBLSVerifierCache, points96: bytes) -> bytes:
    n = len(points96) // 96
    out = (C.c_uint8 * (48 * n))()
    _check(lib().blsgpu_pubkeys_to_bytes(cache.handle, points96, n, out), "pubkeys_to_bytes", cache)
    return bytes(out)


def signaturesToBytes(cache: BatchedBLSVerifierCache, points192: bytes) -> bytes:
    n = len(points192) // 192
    out = (C.c_uint8 * (96 * n))()
    _check(lib().blsgpu_signatures_to_bytes(cache.handle, points192, n, out), "signatures_to_bytes", cache)
    return bytes(out)
