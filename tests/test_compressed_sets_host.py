"""CPU: host side of batch verification on compressed signature sets — the 224-byte record, the scalar-chunk rule of
batchVerify, empty input without a device call, and the declarations the C header and the Nim shim carry."""
import os
import re

import nim_blscurve_b200 as bg

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_compressed_set_packing():
    s = bg.SignatureSetCompressed(b"\x01" * 96, b"\x02" * 32, b"\x03" * 96)
    b = s.to_bytes()
    assert len(b) == 224 and b[:96] == b"\x01" * 96 and b[96:128] == b"\x02" * 32 and b[128:] == b"\x03" * 96
    h = open(os.path.join(ROOT, "include", "blsgpu.h")).read()
    assert re.search(r"#define BLSGPU_COMPRESSED_SET_BYTES 224\b", h)


class FakeCache:
    def __init__(self):
        self.calls = []

    def verify_compressed_raw(self, sets, srb, chunks, scalars=None, want_gt=False):
        self.calls.append((len(sets) // 224, chunks, sets))
        return True, [0] * (len(sets) // 224)


def test_chunk_rule_and_empty_input():
    s = bg.SignatureSetCompressed(b"\x01" * 96, b"\x02" * 32, b"\x03" * 96)
    c = FakeCache()
    tp4, tp1 = bg.Taskpool.new(numThreads=4), bg.Taskpool.new(numThreads=1)
    assert bg.batchVerifyCompressed(tp4, c, [s] * 3, b"\0" * 32) == (True, [0] * 3)    # parallel derivation
    assert bg.batchVerifyCompressed(tp4, c, [s] * 2, b"\0" * 32) == (True, [0] * 2)    # serial: len < 3
    assert bg.batchVerifyCompressed(tp1, c, [tuple(s)] * 5, b"\0" * 32) == (True, [0] * 5)   # serial: one thread
    assert [(n, ch) for n, ch, _ in c.calls] == [(3, 4), (2, 0), (5, 0)]
    assert c.calls[2][2] == s.to_bytes() * 5
    assert bg.batchVerifyCompressed(tp4, c, [], b"\0" * 32) == (False, [])
    assert bg.batchVerifyCompressed(tp4, c, b"", b"\0" * 32) == (False, [])
    assert len(c.calls) == 3


def test_nim_shim_declares_the_compressed_set():
    src = open(os.path.join(ROOT, "nim_blscurve_b200", "nim", "blscurve", "cuda", "bls_batch_verifier_cuda.nim")).read()
    assert re.search(r"SignatureSetCompressed\* = tuple\[pubkey: PublicKey, message: array\[32, byte\], "
                     r"signature: array\[96, byte\]\]", src)
    assert "doAssert sizeof(SignatureSetCompressed) == 224" in src
    assert re.search(r"proc batchVerifyCompressed\*\(\s*tp: Taskpool,\s*cache: var BatchedBLSVerifierCache,\s*"
                     r"input: openArray\[SignatureSetCompressed\],\s*secureRandomBytes: array\[32, byte\],\s*"
                     r"status: var openArray\[byte\]\s*\): bool", src)
