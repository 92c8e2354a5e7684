# blscurve/cuda/blsgpu_abi.nim — FFI declarations of libblsgpu.so (include/blsgpu.h).
#
# Same idioms as blscurve/blst/blst_abi.nim (importc, cdecl, raw pointers, `bool`-like cint results):
# NOT compiled in the build container (no Nim toolchain there); kept in-tree as the reference-side binding
# a maintainer adds.  tests/test_abi_and_host.py parses this file and diffs every proc (name, arity, parameter and
# result types) against include/blsgpu.h, so the two cannot drift apart silently.  See INTEGRATION.md.
{.push raises: [].}

const blsgpuLib* {.strdefine.} = "libblsgpu.so"

type
  BlsGpuCtx* = distinct pointer

{.push cdecl, dynlib: blsgpuLib, importc.}
proc blsgpu_device_count*(): cint
proc blsgpu_create*(device: cint, maxSets: csize_t): BlsGpuCtx
proc blsgpu_create_multi*(devices: ptr cint, ndev: cint, maxSets: csize_t): BlsGpuCtx
proc blsgpu_device_span*(ctx: BlsGpuCtx): cint
proc blsgpu_destroy*(ctx: BlsGpuCtx)
proc blsgpu_last_error*(ctx: BlsGpuCtx): cstring
proc blsgpu_capacity*(ctx: BlsGpuCtx): csize_t
proc blsgpu_set_stream*(ctx: BlsGpuCtx, cudaStream: pointer): cint
proc blsgpu_rlc_scalars*(ctx: BlsGpuCtx, srb: ptr array[32, byte], n: csize_t, chunks: uint32,
                         dst: ptr uint64): cint
proc blsgpu_batch_verify*(ctx: BlsGpuCtx, sets: pointer, n: csize_t, srb: ptr array[32, byte],
                          chunks: uint32, scalars: ptr uint64, gtOut: ptr array[576, byte]): cint
proc blsgpu_batch_verify_compressed*(ctx: BlsGpuCtx, sets: pointer, n: csize_t, srb: ptr array[32, byte],
                                     chunks: uint32, scalars: ptr uint64, gtOut: ptr array[576, byte],
                                     status: ptr byte): cint
proc blsgpu_batch_verify_dev*(ctx: BlsGpuCtx, dSets: pointer, n: csize_t, srb: ptr array[32, byte],
                              chunks: uint32, scalars: ptr uint64, gtOut: ptr array[576, byte]): cint
proc blsgpu_partial*(ctx: BlsGpuCtx, sets: pointer, setsOnDevice: cint, n, first, totalN: csize_t,
                     srb: ptr array[32, byte], chunks: uint32, scalars: ptr uint64,
                     partialOut: ptr array[576, byte], flags: ptr cint): cint
proc blsgpu_partial_dev*(ctx: BlsGpuCtx, dSets: pointer, n, first, totalN: csize_t, srb: ptr array[32, byte],
                         chunks: uint32, dPartialOut: pointer, dFlagOut: ptr cint): cint
proc blsgpu_finalize*(ctx: BlsGpuCtx, partials: ptr byte, count: csize_t, gtOut: ptr array[576, byte]): cint
proc blsgpu_finalize_dev*(ctx: BlsGpuCtx, dPartials: pointer, count: csize_t, dFlags: ptr cint,
                          gtOut: ptr array[576, byte]): cint
proc blsgpu_hash_to_g2*(ctx: BlsGpuCtx, msgs: ptr byte, n, msgLen: csize_t, dst: ptr byte, dstLen: csize_t,
                        outCompressed, outAffine: ptr byte): cint
proc blsgpu_aggregate_g1*(ctx: BlsGpuCtx, points: pointer, n: csize_t, dst: pointer): cint
proc blsgpu_aggregate_g2*(ctx: BlsGpuCtx, points: pointer, n: csize_t, dst: pointer): cint
proc blsgpu_subtract_g1*(ctx: BlsGpuCtx, dst: pointer, elems: pointer, n: csize_t): cint
proc blsgpu_subtract_g2*(ctx: BlsGpuCtx, dst: pointer, elems: pointer, n: csize_t): cint
proc blsgpu_msm_g1*(ctx: BlsGpuCtx, points, scalars: pointer, n, nbits: csize_t, dst: pointer): cint
proc blsgpu_msm_g2*(ctx: BlsGpuCtx, points, scalars: pointer, n, nbits: csize_t, dst: pointer): cint
proc blsgpu_aggregate_g1_segments*(ctx: BlsGpuCtx, points: pointer, offsets: ptr uint32, nseg: csize_t,
                                   dst: pointer): cint
proc blsgpu_aggregate_verify*(ctx: BlsGpuCtx, pubkeys: pointer, n: csize_t, msgs: ptr byte, msgOffsets: ptr uint32,
                              dst: ptr byte, dstLen: csize_t, sig: pointer, gtOut: ptr array[576, byte]): cint
proc blsgpu_fast_aggregate_verify*(ctx: BlsGpuCtx, pubkeys: pointer, n: csize_t, msg: ptr byte, msgLen: csize_t,
                                   dst: ptr byte, dstLen: csize_t, sig: pointer, gtOut: ptr array[576, byte]): cint
proc blsgpu_pubkeys_from_bytes*(ctx: BlsGpuCtx, raw: ptr byte, n, inLen: csize_t, groupCheck: cint,
                                dst: pointer, status: ptr byte): cint
proc blsgpu_signatures_from_bytes*(ctx: BlsGpuCtx, raw: ptr byte, n, inLen: csize_t, groupCheck: cint,
                                   dst: pointer, status: ptr byte): cint
proc blsgpu_pubkeys_to_bytes*(ctx: BlsGpuCtx, points: pointer, n: csize_t, dst: ptr byte): cint
proc blsgpu_signatures_to_bytes*(ctx: BlsGpuCtx, points: pointer, n: csize_t, dst: ptr byte): cint
proc blsgpu_combine*(ctx: BlsGpuCtx, srb: ptr array[32, byte], pubkeys, sigs: pointer, n: csize_t,
                     pkOut, sigOut: pointer): cint
proc blsgpu_msm_g1_dev*(ctx: BlsGpuCtx, dPoints, dScalars: pointer, n, nbits: csize_t, dst: pointer): cint
proc blsgpu_msm_g2_dev*(ctx: BlsGpuCtx, dPoints, dScalars: pointer, n, nbits: csize_t, dst: pointer): cint
proc blsgpu_last_stage_ms*(ctx: BlsGpuCtx, ms: ptr cfloat, max: cint): cint
proc blsgpu_stage_name*(stage: cint): cstring
proc blsgpu_last_launches*(ctx: BlsGpuCtx): cint
# diagnostics / synthetic workloads (benchmarks and tests only)
proc blsgpu_test_fp*(ctx: BlsGpuCtx, op: cint, a, b: pointer, n: csize_t, dst: pointer): cint
proc blsgpu_test_field*(ctx: BlsGpuCtx, op: cint, src: pointer, inRecBytes, n: csize_t, dst: pointer,
                        outRecBytes: csize_t): cint
proc blsgpu_test_small_hash*(ctx: BlsGpuCtx, sets: pointer, n: csize_t, outIn, outOut: ptr byte): cint
proc blsgpu_imad_peak*(ctx: BlsGpuCtx, wide: cint): cdouble
proc blsgpu_fpmul_peak*(ctx: BlsGpuCtx, threadsPerBlock, blocksPerSm: cint): cdouble
proc blsgpu_make_sets*(ctx: BlsGpuCtx, seed: uint64, first, n: csize_t, dst: pointer, outOnDevice: cint): cint
proc blsgpu_msm_make_inputs*(ctx: BlsGpuCtx, seed: uint64, n: csize_t, dPoints, dScalars: pointer): cint
{.pop.}
{.pop.}
