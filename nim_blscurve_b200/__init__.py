"""B200-native batch BLS12-381 signature verification behind the nim-blscurve batch-verifier API.

Host-side mirror (Python, over the C ABI of libblsgpu.so) of
  blscurve/bls_batch_verifier.nim : SignatureSet, MultiSignatureSet, BatchedBLSVerifierCache,
                                    batchVerifySerial, batchVerifyParallel, batchVerify
  blscurve/blst/blst_min_pubkey_sig_core.nim : aggregateAll, subtractAll
plus the companion G1 MSM.  All arithmetic runs in hand-written sm_100a CUDA kernels
(nim_blscurve_b200/csrc); there is no CPU fallback.
"""
from ._lib import BlsGpuError, LIB_PATH, lib  # noqa: F401
from .batch_verifier import (  # noqa: F401
    BatchedBLSVerifierCache, MultiSignatureSet, SignatureSet, SignatureSetCompressed, Taskpool, batchVerifyCompressed, aggregateAll, combine, batchVerify, batchVerifyParallel,
    batchVerifySerial, hashToG2, msmG1, msmG2, rlcScalars, aggregateVerify, verify, fastAggregateVerify, aggregateAllSegments, subtractAll,
    publicKeysFromBytes, signaturesFromBytes, publicKeysToBytes, signaturesToBytes,
)
from .multi_gpu import GpuBackend, batch_verify_distributed, msm_g1_distributed, shard_range  # noqa: F401,E402
