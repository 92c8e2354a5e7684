# blscurve/cuda/bls_batch_verifier_cuda.nim — drop-in bodies for blscurve/bls_batch_verifier.nim on libblsgpu.so.
#
# Every public name, parameter list and result below is the reference's (file:line into nim-blscurve):
#   SignatureSet :34, MultiSignatureSet :47 (+ init :73/:86, add :93, combine :100), BatchedBLSVerifierCache :62,
#   init :108 / :115, batchVerifySerial :121 / :162, batchVerifyParallel :296 (ptr) / :373 / :399,
#   batchVerify :420 (ptr) / :449 / :475;
#   aggregateAll / subtractAll (blst_min_pubkey_sig_core.nim:179, :197) and combine (:570) keep their cache-less
#   signatures through a lazily created per-thread context.
# `tp: Taskpool` stays in the signatures; it no longer fans work out — tp.numThreads only selects the reference's
# RLC-scalar chunking (numBatches = min(numSets, tp.numThreads), :316), so verdicts (and GT values) are identical to
# the BLST path for the same tp.  The fan-out itself happens on the device(s): `-d:blsgpuNumDevices=N` makes every
# cache span N GPUs (0 = all visible) through blsgpu_create_multi — one call, N shares, one final exponentiation.
#
# Error convention: the reference returns one `bool` and asserts on misuse (:141, :319).  Here 1 -> true, 0 -> false,
# and a NEGATIVE code (CUDA failure, bad argument) is a Defect carrying blsgpu_last_error — it is never reported as an
# invalid signature.  There is no CPU fallback: without a CUDA device the first use asserts.
#
# NOT compiled in the build container (no Nim toolchain there); tests/test_abi_and_host.py checks the FFI declarations
# against include/blsgpu.h mechanically and the overload set against the reference's.  See INTEGRATION.md.
{.push raises: [].}

import taskpools
import ../blst/blst_min_pubkey_sig_core   # PublicKey, Signature (in-memory blst_p1_affine / blst_p2_affine)
import ./blsgpu_abi

const
  blsgpuDefaultSets* {.intdefine.} = 16384   ## initial capacity of a cache; grows on demand
  blsgpuNumDevices* {.intdefine.} = 1        ## GPUs one cache spans (0 = all visible devices)
  blsgpuDevice* {.intdefine.} = 0            ## first device index

type
  SignatureSet* = tuple[pubkey: PublicKey, message: array[32, byte], signature: Signature]

  SignatureSetCompressed* = tuple[pubkey: PublicKey, message: array[32, byte], signature: array[96, byte]]
    ## a set as it comes off the network: the signature still in its Zcash compressed encoding (bls_sig_io.nim:20-36)

  MultiSignatureSet* = object                                # bls_batch_verifier.nim:47-62
    pubkeys: seq[PublicKey]
    message: array[32, byte]
    signatures: seq[Signature]

  BatchedBLSVerifierCache* {.requiresInit.} = object
    ## device scratch instead of per-thread pairing contexts (:62-69); reusable across calls
    ctx: BlsGpuCtx
    numThreads: int

static: doAssert sizeof(SignatureSet) == 320   # pk 96 | msg 32 | sig 192, no padding
static: doAssert sizeof(SignatureSetCompressed) == 224   # pk 96 | msg 32 | compressed sig 96, no padding

# ---- context lifetime --------------------------------------------------------------------------------------
proc createCtx(maxSets: int): BlsGpuCtx =
  ## one device, or a multi-device context behind the same handle
  let visible = blsgpu_device_count().int
  doAssert visible > 0, "libblsgpu: no CUDA device visible (there is no CPU fallback)"
  let want = if blsgpuNumDevices <= 0: visible else: min(blsgpuNumDevices, visible)
  if want <= 1:
    result = blsgpu_create(blsgpuDevice.cint, maxSets.csize_t)
  else:
    var devices: array[64, cint]
    for k in 0 ..< min(want, 64): devices[k] = cint((blsgpuDevice + k) mod visible)
    result = blsgpu_create_multi(addr devices[0], min(want, 64).cint, maxSets.csize_t)
  doAssert not pointer(result).isNil, "blsgpu_create failed: " & $blsgpu_last_error(BlsGpuCtx(nil))

proc `=destroy`(c: var BatchedBLSVerifierCache) =
  if not pointer(c.ctx).isNil:
    blsgpu_destroy(c.ctx)
    c.ctx = BlsGpuCtx(nil)

proc `=copy`(dst: var BatchedBLSVerifierCache, src: BatchedBLSVerifierCache) {.error:
  "a BatchedBLSVerifierCache owns a device context: move it or create another one".}

proc ensureCapacity(ctx: var BlsGpuCtx, n: int) =
  ## the reference has no size limit: grow instead of failing (destroy + re-create at the next power of two)
  if pointer(ctx).isNil or blsgpu_capacity(ctx).int < n:
    var cap = max(blsgpuDefaultSets, 1)
    while cap < n: cap = cap * 2
    if not pointer(ctx).isNil: blsgpu_destroy(ctx)
    ctx = createCtx(cap)

func init*(T: type BatchedBLSVerifierCache): T =
  ## Initialise the cache for single-threaded usage (:108-113)
  {.cast(noSideEffect).}:
    result = T(ctx: createCtx(blsgpuDefaultSets), numThreads: 1)

when compileOption("threads"):
  func init*(T: type BatchedBLSVerifierCache, tp: Taskpool): T =
    ## Initialise the cache for multi-threaded usage (:115-119)
    {.cast(noSideEffect).}:
      result = T(ctx: createCtx(blsgpuDefaultSets), numThreads: tp.numThreads)

# A lazily created context per host thread for the cache-less entry points (batchVerifySerial(input, srb) :162,
# batchVerifyParallel(tp, input, srb) :399, batchVerify(tp, input, srb) :475, aggregateAll, subtractAll, combine).
# The reference builds a throw-away cache per call there; a device context is too heavy for that.
var tlsCtx {.threadvar.}: BlsGpuCtx

proc threadCtx(n: int): BlsGpuCtx =
  ensureCapacity(tlsCtx, n)
  tlsCtx

proc check(ctx: BlsGpuCtx, rc: cint, what: string): bool =
  ## 1 / 0 are the reference's booleans; anything negative is a runtime failure, never "invalid signature"
  doAssert rc >= 0, what & " failed (" & $rc & "): " & $blsgpu_last_error(ctx)
  rc == 1

proc verifyRaw(ctx: var BlsGpuCtx, sets: ptr UncheckedArray[SignatureSet], n: int,
               srb: ptr array[32, byte], chunks: uint32): bool =
  if n == 0: return false                                    # spec precondition (:137, :312)
  ensureCapacity(ctx, n)
  check(ctx, blsgpu_batch_verify(ctx, sets, n.csize_t, srb, chunks, nil, nil), "blsgpu_batch_verify")

# ---- serial batch verifier (:121-165) ---------------------------------------------------------------------
func batchVerifySerial*(
       cache: var BatchedBLSVerifierCache,
       input: openArray[SignatureSet],
       secureRandomBytes: array[32, byte]
     ): bool =
  if input.len == 0: return false
  {.cast(noSideEffect).}:
    result = cache.ctx.verifyRaw(cast[ptr UncheckedArray[SignatureSet]](unsafeAddr input[0]), input.len,
                                 unsafeAddr secureRandomBytes, 0'u32)

func batchVerifySerial*(
       input: openArray[SignatureSet],
       secureRandomBytes: array[32, byte]
     ): bool =
  if input.len == 0: return false
  {.cast(noSideEffect).}:
    discard threadCtx(input.len)
    result = tlsCtx.verifyRaw(cast[ptr UncheckedArray[SignatureSet]](unsafeAddr input[0]), input.len,
                              unsafeAddr secureRandomBytes, 0'u32)

# ---- parallel batch verifier (:296-403) -------------------------------------------------------------------
when compileOption("threads"):
  proc batchVerifyParallel*(
        tp: Taskpool,
        cache: ptr BatchedBLSVerifierCache,
        setsPtr: ptr UncheckedArray[SignatureSet],
        numSets: int,
        secureRandomBytes: ptr array[32, byte]
      ): bool {.sideEffect.} =
    ## the form a threaded consumer (nimbus-eth2) calls; does not allocate garbage-collected memory
    if numSets == 0: return false
    cache[].ctx.verifyRaw(setsPtr, numSets, secureRandomBytes, uint32 max(1, tp.numThreads))

  proc batchVerifyParallel*(
        tp: Taskpool,
        cache: var BatchedBLSVerifierCache,
        input: openArray[SignatureSet],
        secureRandomBytes: array[32, byte]
      ): bool {.sideEffect.} =
    if input.len == 0: return false
    batchVerifyParallel(tp, addr cache, cast[ptr UncheckedArray[SignatureSet]](unsafeAddr input[0]), input.len,
                        unsafeAddr secureRandomBytes)

  proc batchVerifyParallel*(
        tp: Taskpool,
        input: openArray[SignatureSet],
        secureRandomBytes: array[32, byte]
      ): bool =
    if input.len == 0: return false
    discard threadCtx(input.len)
    tlsCtx.verifyRaw(cast[ptr UncheckedArray[SignatureSet]](unsafeAddr input[0]), input.len,
                     unsafeAddr secureRandomBytes, uint32 max(1, tp.numThreads))

  # ---- autoselect (:420-495): parallel derivation iff tp.numThreads > 1 and numSets >= 3 ------------------
  proc batchVerify*(
        tp: Taskpool,
        cache: ptr BatchedBLSVerifierCache,
        setsPtr: ptr UncheckedArray[SignatureSet],
        numSets: int,
        secureRandomBytes: ptr array[32, byte]
      ): bool =
    if tp.numThreads > 1 and numSets >= 3:
      tp.batchVerifyParallel(cache, setsPtr, numSets, secureRandomBytes)
    else:
      if numSets == 0: return false
      cache[].ctx.verifyRaw(setsPtr, numSets, secureRandomBytes, 0'u32)

  proc batchVerify*(
        tp: Taskpool,
        cache: var BatchedBLSVerifierCache,
        input: openArray[SignatureSet],
        secureRandomBytes: array[32, byte]
      ): bool =
    if tp.numThreads > 1 and input.len >= 3:
      tp.batchVerifyParallel(cache, input, secureRandomBytes)
    else:
      cache.batchVerifySerial(input, secureRandomBytes)

  proc batchVerify*(
        tp: Taskpool,
        input: openArray[SignatureSet],
        secureRandomBytes: array[32, byte]
      ): bool =
    if tp.numThreads > 1 and input.len >= 3:
      tp.batchVerifyParallel(input, secureRandomBytes)
    else:
      batchVerifySerial(input, secureRandomBytes)

  # ---- Signature.fromBytes (bls_sig_io.nim:42-60) of every set + batchVerify, decoded and checked on the device -----
  proc batchVerifyCompressed*(
        tp: Taskpool,
        cache: var BatchedBLSVerifierCache,
        input: openArray[SignatureSetCompressed],
        secureRandomBytes: array[32, byte],
        status: var openArray[byte]
      ): bool =
    ## status[i] receives the BLST_ERROR of signature i (0 success, 1 bad encoding, 2 not on curve, 3 not in group);
    ## any failure makes the batch false.  Scalar chunking as batchVerify (:420-495).
    doAssert status.len == input.len
    if input.len == 0: return false
    ensureCapacity(cache.ctx, input.len)
    let chunks = if tp.numThreads > 1 and input.len >= 3: uint32 tp.numThreads else: 0'u32
    check(cache.ctx, blsgpu_batch_verify_compressed(cache.ctx, unsafeAddr input[0], input.len.csize_t,
                                                    unsafeAddr secureRandomBytes, chunks, nil, nil, addr status[0]),
          "blsgpu_batch_verify_compressed")

# ---- MultiSignatureSet (:73-106) --------------------------------------------------------------------------
func init*(
       T: type MultiSignatureSet,
       pubkeys: seq[PublicKey],
       message: array[32, byte],
       signatures: seq[Signature]
     ): MultiSignatureSet =
  doAssert pubkeys.len == signatures.len
  doAssert pubkeys.len > 0
  MultiSignatureSet(pubkeys: pubkeys, message: message, signatures: signatures)

func init*(T: type MultiSignatureSet, sigset: SignatureSet): MultiSignatureSet =
  MultiSignatureSet(pubkeys: @[sigset.pubkey], message: sigset.message, signatures: @[sigset.signature])

func add*(multiSet: var MultiSignatureSet, sigset: SignatureSet) =
  doAssert multiSet.message == sigset.message
  multiSet.pubkeys.add sigset.pubkey
  multiSet.signatures.add sigset.signature

func combine*(
         secureRandomBytes: array[32, byte],
         publicKeys: openArray[PublicKey],
         signatures: openArray[Signature],
       ): tuple[publicKey: PublicKey, signature: Signature] =
  ## blst_min_pubkey_sig_core.nim:570-647 on the device: the reference's scalar order, two 64-bit Pippenger MSMs
  doAssert publicKeys.len == signatures.len
  if publicKeys.len == 0:
    raiseAssert "Must provide at least 1 signature"
  if publicKeys.len == 1:
    return (publicKeys[0], signatures[0])
  {.cast(noSideEffect).}:
    let ctx = threadCtx(1)
    let rc = blsgpu_combine(ctx, unsafeAddr secureRandomBytes, unsafeAddr publicKeys[0], unsafeAddr signatures[0],
                            publicKeys.len.csize_t, addr result.publicKey, addr result.signature)
    doAssert check(ctx, rc, "blsgpu_combine")

func combine*(
          multiSet: MultiSignatureSet,
          secureRandomBytes: array[32, byte]
        ): SignatureSet =
  ## bls_batch_verifier.nim:100-106
  let (pubkey, signature) = secureRandomBytes.combine(multiSet.pubkeys, multiSet.signatures)
  (pubkey, multiSet.message, signature)

# ---- aggregateAll / subtractAll (blst_min_pubkey_sig_core.nim:179-209), reference signatures ----------------
proc aggregateAll*(dst: var PublicKey, elems: openArray[PublicKey]): bool =
  if elems.len == 0: return false                            # :183-184
  let ctx = threadCtx(1)
  check(ctx, blsgpu_aggregate_g1(ctx, unsafeAddr elems[0], elems.len.csize_t, addr dst), "blsgpu_aggregate_g1")

proc aggregateAll*(dst: var Signature, elems: openArray[Signature]): bool =
  if elems.len == 0: return false
  let ctx = threadCtx(1)
  check(ctx, blsgpu_aggregate_g2(ctx, unsafeAddr elems[0], elems.len.csize_t, addr dst), "blsgpu_aggregate_g2")

proc subtractAll*(dst: var PublicKey, elems: openArray[PublicKey]) =
  ## dst <- dst - sum(elems)                                   # :197-209
  if elems.len == 0: return
  let ctx = threadCtx(1)
  doAssert check(ctx, blsgpu_subtract_g1(ctx, addr dst, unsafeAddr elems[0], elems.len.csize_t), "blsgpu_subtract_g1")

proc subtractAll*(dst: var Signature, elems: openArray[Signature]) =
  if elems.len == 0: return
  let ctx = threadCtx(1)
  doAssert check(ctx, blsgpu_subtract_g2(ctx, addr dst, unsafeAddr elems[0], elems.len.csize_t), "blsgpu_subtract_g2")

# ---- SURVEY §8f N3: bls_sig_min_pubkey.nim:108-258 on the device (the proof-of-possession overloads stay as they
# are: they call popVerify per key and then these).  Named *Cuda: the BLST forms remain the default for one pairing
# check (INTEGRATION.md section 7), a consumer opts in per call site. ---
const DST = "BLS_SIG_BLS12381G2_XMD:SHA-256_SSWU_RO_POP_"        # bls_sig_min_pubkey.nim:31

proc verifyCuda*[T: byte|char](publicKey: PublicKey, message: openArray[T], signature: Signature): bool =
  ## coreVerifyNoGroupCheck (blst_min_pubkey_sig_core.nim:264-297) = aggregateVerify over one pair
  var offs = [0'u32, uint32 message.len]
  let ctx = threadCtx(1)
  check(ctx, blsgpu_aggregate_verify(ctx, unsafeAddr publicKey, 1,
                                     (if message.len > 0: cast[ptr byte](unsafeAddr message[0]) else: nil),
                                     addr offs[0], cast[ptr byte](unsafeAddr DST[0]), DST.len.csize_t,
                                     unsafeAddr signature, nil), "blsgpu_aggregate_verify")

proc fastAggregateVerifyCuda*[T: byte|char](publicKeys: openArray[PublicKey], message: openArray[T],
                                            signature: Signature): bool =
  if publicKeys.len == 0: return false                       # :251-253
  let ctx = threadCtx(1)
  check(ctx, blsgpu_fast_aggregate_verify(ctx, unsafeAddr publicKeys[0], publicKeys.len.csize_t,
                                          (if message.len > 0: cast[ptr byte](unsafeAddr message[0]) else: nil),
                                          message.len.csize_t, cast[ptr byte](unsafeAddr DST[0]), DST.len.csize_t,
                                          unsafeAddr signature, nil), "blsgpu_fast_aggregate_verify")

proc aggregateVerifyCuda*(publicKeys: openArray[PublicKey], messages: openArray[seq[byte]],
                          signature: Signature): bool =
  if publicKeys.len != messages.len or publicKeys.len < 1: return false     # :164-169
  var blob: seq[byte]
  var offs = newSeq[uint32](messages.len + 1)
  for i, m in messages:
    blob.add m
    offs[i + 1] = uint32 blob.len
  let ctx = threadCtx(publicKeys.len)
  check(ctx, blsgpu_aggregate_verify(ctx, unsafeAddr publicKeys[0], publicKeys.len.csize_t,
                                     (if blob.len > 0: addr blob[0] else: nil), addr offs[0],
                                     cast[ptr byte](unsafeAddr DST[0]), DST.len.csize_t, unsafeAddr signature, nil),
        "blsgpu_aggregate_verify")

# ---- SURVEY §8f N2: bls_sig_io.nim:42-122, batched ---------------------------------------------------------
proc fromBytesBatch*(dst: var openArray[PublicKey], raw: openArray[array[48, byte]], ok: var openArray[bool]): bool =
  ## every element as PublicKey.fromBytes: uncompress, reject infinity, subgroup check
  doAssert dst.len == raw.len and ok.len == raw.len
  if raw.len == 0: return true
  var status = newSeq[byte](raw.len)
  let ctx = threadCtx(1)
  result = check(ctx, blsgpu_pubkeys_from_bytes(ctx, cast[ptr byte](unsafeAddr raw[0]), raw.len.csize_t, 48, 1,
                                                addr dst[0], addr status[0]), "blsgpu_pubkeys_from_bytes")
  for i in 0 ..< raw.len: ok[i] = status[i] == 0

proc fromBytesBatch*(dst: var openArray[Signature], raw: openArray[array[96, byte]], ok: var openArray[bool]): bool =
  doAssert dst.len == raw.len and ok.len == raw.len
  if raw.len == 0: return true
  var status = newSeq[byte](raw.len)
  let ctx = threadCtx(1)
  result = check(ctx, blsgpu_signatures_from_bytes(ctx, cast[ptr byte](unsafeAddr raw[0]), raw.len.csize_t, 96, 1,
                                                   addr dst[0], addr status[0]), "blsgpu_signatures_from_bytes")
  for i in 0 ..< raw.len: ok[i] = status[i] == 0
{.pop.}
