#!/usr/bin/env python3
"""bench.py — batch-verified signature sets/s on N B200 (one process per GPU).

Workload (config.workload): the per-GPU share of BASELINE.json configs[4] — "1M distinct-message signature
sets on 8xB200" = 131,072 sets per GPU (weak scaling: N GPUs verify ONE batch of N*131,072 sets).  A step is
one batch verification: every rank runs the per-set pipeline on its share (RLC scalars, hash_to_G2, [r]pk,
[r]sig, Miller loops, GT product), emits one 576-byte Fp12 partial, NCCL all-gathers the partials (ONE
collective: a share that must fail the batch seals its partial as zero) and ONE final exponentiation decides.

The RLC scalars are derived exactly as the drop-in derives them: `rlc_chunks` = tp.numThreads of the caller =
the host's hardware threads (--chunks; the same thread count the reference arm runs with), i.e. a handful of
long sequential SHA-256 chains — not a benchmark-friendly chunk count.

  value  : sets/s with the sets resident in HBM (device-generated synthetic valid sets, distinct messages)
  e2e    : the plugin call itself — blsgpu_batch_verify(host buffer) at N = 1 (pinned buffer; the pageable figure
           beside it), per-rank H2D + blsgpu_partial_dev + NCCL + blsgpu_finalize_dev at N > 1
  --impl reference : the reference's own CPU path (BLST from oracle/_ref driven by oracle/ref_batch.c, the
                     pthreads replica of batchVerifyParallel) on all host cores, on the first n sets of the SAME
                     workload (bounded sample per step).
Extras on the same JSON line (rank 0): config1 (BASELINE configs[0], 64 sets), block_batch (configs[1]),
msm_g1 (configs[2], 2^20 headline + sweep 2^16..2^22), config3 (32,768 sets over the N ranks), streaming_blocks
(K contexts in flight), batch_sizes, chunk_sweep, parity_checks.
"""
import argparse
import ctypes as C
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SETS_PER_GPU = 131072
SEED = 2026
W_SET = 12725                  # Fp-mul per set of the reference algorithm (SURVEY.md §8a/d)
W_BATCH = 14673                # per batch finalisation
IMAD_PER_FPMUL = 300
# reference-algorithm Fp-mul per set of each stage (SURVEY.md §8a): A3, A5 (G1), A4, and A7 split into its line
# evaluations (63 x (25+4) + 5 x (35+4)) and its accumulation (68 x 39 + shared squarings)
STAGE_FPMUL = {"hash_to_g2": 4919, "g1_mul64": 800, "pairs_affine": 23, "miller_lines": 2022, "miller_acc": 2933}
# algorithmic bytes per set moved by each stage's kernel (inputs read + outputs written; DESIGN.md section 3)
STAGE_IO_BYTES = {"hash_to_g2": 32 + 288, "g1_mul64": 96 + 8 + 144, "miller_lines": 192 + 96 + 68 * 288,
                  "miller_acc": 68 * 288 + 576 // 8}
STAGE_KERNEL = {"hash_to_g2": "k_hash_sets", "miller_lines": "k_miller_lines", "miller_acc": "k_miller_acc_team",
                "g1_mul64": "k_g1_mul"}
# IMAD.WIDE warp-instructions x 32 lanes EXECUTED per set by each kernel (ncu source page of the committed capture of
# the same workload, profiles/): the numerator of roofline.frac_executed
EXECUTED_IMAD_WIDE_PER_SET = {"hash_to_g2": 5099991040 * 32 / 131072}


def host_threads():
    return os.cpu_count() or 1


def default_chunks(world):
    """RLC chunk count of the headline run = tp.numThreads of the caller: the host's hardware threads, and at least 16 per
    GPU (a host that feeds N GPUs with N shares brings N x 16 threads' worth of chunks; the sequential SHA-256 chain of a
    chunk — total/chunks blocks, ~2 us each on the device — is the one part of the path that does not shrink with N)."""
    return max(host_threads(), 16 * world)


def make_config(S, world, chunks):
    """One dict for both arms (the driver compares them)."""
    total = S * world
    return {"workload": f"{S} distinct-message signature sets per GPU = per-GPU share of BASELINE configs[4] "
                        f"(1M sets on 8 GPUs); one batch of {total} sets per step; sets = blsgpu_make_sets(seed {SEED})",
            "sets_per_step": total, "rlc_chunks": chunks,
            "rlc_chunks_note": "tp.numThreads the drop-in passes: max(host hardware threads, 16 per GPU); chunk_sweep has 0 / 16 / 64 / 1024",
            "l2": "GPU arm: 256 MiB flush write between steps",
            "partial_exchange": "NCCL all_gather of one 576-byte Fp12 per rank (one collective per step)" if world > 1 else "none"}


def clocks_sampler(stop, out, gpu_index):
    q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
    while not stop.is_set():
        try:
            r = subprocess.run(["nvidia-smi", "-i", str(gpu_index), f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                               capture_output=True, text=True, timeout=5)
            f = [x.strip() for x in r.stdout.strip().split(",")]
            if len(f) >= 6:
                out.append(f)
        except Exception:
            pass
        stop.wait(0.2)


def summarize_clocks(samples):
    if not samples:
        return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
    sm = sorted(int(s[0]) for s in samples if s[0].isdigit())
    names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
    reasons = [n for i, n in enumerate(names) if any(s[2 + i].lower().startswith("active") for s in samples)]
    return {"sm_mhz": sm[len(sm) // 2] if sm else None,
            "sm_max_mhz": int(samples[0][1]) if samples[0][1].isdigit() else None, "reasons": reasons}


def run_reference(args):
    """The reference's CPU implementation of the path on this host's cores (rank 0 only), on the first n sets of the
    SAME workload the GPU arm verifies (oracle ref_make_sets_device_recipe = blsgpu_make_sets on the host)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    from oracle import blst_ref as br
    cores = br.ncores()
    world = int(os.environ.get("WORLD_SIZE", str(args.gpus)))
    S = args.sets_per_gpu
    chunks = args.chunks if args.chunks >= 0 else default_chunks(world)
    srb = hashlib.sha256(b"Mr F was here").digest()
    n = max(64, min(S * world, 1200 * cores))              # ~1-2 s of CPU work per step
    sets = br.make_sets_device_recipe(SEED, 0, n)          # first n sets of the timed workload, all distinct
    for _ in range(max(args.warmup, 1)):
        assert br.batch_verify_mt(sets, srb, cores)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        ok = br.batch_verify_mt(sets, srb, cores)
        assert ok
    dt = time.perf_counter() - t0
    v = n * args.steps / dt
    line = {
        "impl": "reference", "metric": "batch-verified signature sets/sec", "value": v, "unit": "sets/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": max(args.warmup, 1), "ms_per_step": dt / args.steps * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u32x12 (Fp 381-bit Montgomery)",
        "data": "synthetic", "gpu_launches": 0,
        "config": make_config(S, world, chunks),
        "sample_sets_per_step": n,
        "cpu_baseline": {"value": v, "unit": "sets/s", "cores": cores, "kind": "reference",
                         "sample": f"first {n} sets of the workload per step (all distinct), BLST batchVerifyParallel "
                                   f"replica (pthreads, {cores} threads = {cores} RLC chunks), {args.steps} steps"},
        "e2e": {"value": v, "unit": "sets/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)
    return 0


def msm_once(L, h, stream, flush, dp, ds, n, reps):
    import torch
    out = (C.c_uint8 * 96)()
    for _ in range(2):
        assert L.blsgpu_msm_g1_dev(h, C.c_void_p(dp.data_ptr()), C.c_void_p(ds.data_ptr()), n, 255, out) == 1
    tot = 0.0
    for _ in range(reps):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        L.blsgpu_msm_g1_dev(h, C.c_void_p(dp.data_ptr()), C.c_void_p(ds.data_ptr()), n, 255, out)
        e1.record(stream)
        torch.cuda.synchronize()
        tot += e0.elapsed_time(e1)
    return tot / reps, bytes(out)


W_PT = {16: 235, 17: 220, 18: 205, 19: 190, 20: 176, 21: 170, 22: 165}     # SURVEY.md §8a A12 (model, Fp-mul per point)


def bench_msm(L, h, stream, flush, peak_wide, hbm_peak, args):
    """BASELINE metric, second half: G1 MSM over 2^20 points, ms (benchmarks/bls12381_msm_g1.nim shape: 96-bit-multiple
    points, 255-bit scalars), plus the sweep 2^16..2^22 of configs[2].  Inputs generated on the device; timed with CUDA
    events on the launching stream, L2 flushed between repetitions.  Roofline: reference-algorithm work W_pt Fp-mul per
    point (SURVEY.md §8a A12) x 300 IMAD against the measured IMAD.WIDE peak; HBM bytes (points + scalars read once) as
    the secondary figure.  CPU beside it: BLST blst_p1s_mult_pippenger, ONE thread (the reference benchmark is
    single-threaded), same inputs — which also makes this a full-size parity check of the affine result (<= 2^20)."""
    import torch
    dev = flush.device
    kmax = max(args.msm_log2, 22 if not args.no_msm_sweep else args.msm_log2)
    nmax = 1 << kmax
    dp = torch.empty(nmax * 96, dtype=torch.uint8, device=dev)
    ds = torch.empty(nmax * 32, dtype=torch.uint8, device=dev)
    assert L.blsgpu_msm_make_inputs(h, 0xFACADE, nmax, C.c_void_p(dp.data_ptr()), C.c_void_p(ds.data_ptr())) == 0
    k = args.msm_log2
    n = 1 << k
    ms, out = msm_once(L, h, stream, flush, dp, ds, n, 5)
    launches = L.blsgpu_last_launches(h)
    # e2e: host points + scalars -> H2D -> MSM -> affine result back
    hp, hs = dp[:n * 96].cpu().pin_memory(), ds[:n * 32].cpu().pin_memory()
    o2 = (C.c_uint8 * 96)()
    assert L.blsgpu_msm_g1(h, C.c_void_p(hp.data_ptr()), C.c_void_p(hs.data_ptr()), n, 255, o2) == 1
    t0 = time.perf_counter()
    for _ in range(3):
        L.blsgpu_msm_g1(h, C.c_void_p(hp.data_ptr()), C.c_void_p(hs.data_ptr()), n, 255, o2)
    ms_e2e = (time.perf_counter() - t0) / 3 * 1e3
    w_pt = W_PT.get(k, 176)
    res = {"metric": "G1 MSM 2^%d points" % k, "value": ms, "unit": "ms", "higher_is_better": False, "n": n, "nbits": 255,
           "points_per_s": n / (ms * 1e-3), "gpu_launches": launches,
           "e2e": {"value": ms_e2e, "unit": "ms", "h2d_bytes": n * 128, "d2h_bytes": 96},
           "roofline": {"bound": "int_mul_pipe", "achieved": n * w_pt * IMAD_PER_FPMUL / (ms * 1e-3) / 1e9,
                        "peak": peak_wide / 1e9, "unit": "G IMAD.WIDE/s",
                        "frac": n * w_pt * IMAD_PER_FPMUL / (ms * 1e-3) / peak_wide,
                        "algorithmic_fpmul_per_point": w_pt,
                        "hbm": {"achieved_gbs": n * 128 / (ms * 1e-3) / 1e9, "peak_gbs": hbm_peak,
                                "note": "points + scalars read once = 128 B/point: not the bound"}}}
    br = None
    if not args.no_cpu_baseline:
        try:
            from oracle import blst_ref as br
        except Exception as ex:
            res["cpu_baseline"] = {"value": None, "unit": "ms", "cores": 0, "kind": "reference", "sample": f"unavailable: {ex}"}
            br = None

    def cpu(kk, expect):
        nn = 1 << kk
        p, s = dp[:nn * 96].cpu().numpy().tobytes(), ds[:nn * 32].cpu().numpy().tobytes()
        ref_out = (C.c_uint8 * 96)()
        t0 = time.perf_counter()
        br.ref.ref_msm_g1(p, s, C.c_size_t(nn), C.c_size_t(255), ref_out)
        return (time.perf_counter() - t0) * 1e3, bytes(ref_out) == expect

    if br is not None:
        tc, same = cpu(k, out)
        res["cpu_baseline"] = {"value": tc, "unit": "ms", "cores": 1, "kind": "reference",
                               "sample": "the same 2^%d inputs, blst_p1s_mult_pippenger + to_affine, one run" % k}
        res["matches_reference"] = same
    if not args.no_msm_sweep:
        sweep = {}
        for kk in range(16, 23):
            if kk == k:
                row = {"ms": ms, "frac": res["roofline"]["frac"]}
                if "matches_reference" in res:
                    row.update({"cpu_ms": res["cpu_baseline"]["value"], "matches_reference": res["matches_reference"]})
            else:
                nn = 1 << kk
                m, o = msm_once(L, h, stream, flush, dp, ds, nn, 3)
                row = {"ms": m, "frac": nn * W_PT[kk] * IMAD_PER_FPMUL / (m * 1e-3) / peak_wide}
                if br is not None and kk <= 19:
                    tc, same = cpu(kk, o)
                    row.update({"cpu_ms": tc, "matches_reference": same})
            sweep["2^%d" % kk] = row
        res["sweep"] = sweep
        res["sweep_note"] = "BASELINE configs[2]: prefixes of one device-generated input set; resident, CUDA events, L2 flushed; " \
                            "cpu_ms = one BLST thread on the same bytes (<= 2^20); 2^21/2^22 are pinned by slice-sum properties " \
                            "in tests/test_gpu_msm.py"
    return res


def ncu_traffic(kernel):
    """DRAM bytes (read + write) of one launch of `kernel` from the committed `ncu --set full` capture of the same
    workload (profiles/r2 if present, else profiles/r1: <round>_raw_pick_<kernel>.txt, tools/gpu_profile.sh)."""
    mult = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9, "Tbyte": 1e12}
    for rnd in ("r2", "r1"):
        path = os.path.join(ROOT, "profiles", rnd, "%s_raw_pick_%s.txt" % (rnd, kernel))
        tot, seen = 0.0, 0
        try:
            for ln in open(path):
                f = ln.split()
                if len(f) >= 3 and f[0] in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
                    tot += float(f[1].replace(",", "")) * mult.get(f[2], 1.0)
                    seen += 1
        except OSError:
            continue
        if seen == 2:
            return tot, os.path.relpath(path, ROOT)
    return None, None


def bench_streaming(L, bg, h_sets_bytes, srb, blk, nctx, batches_each, chunks):
    """K contexts in flight on one GPU, one host thread each, every thread verifying `blk`-set batches back to back
    through blsgpu_batch_verify from its own host buffer (what a node verifying blocks as they arrive does)."""
    caches = [bg.BatchedBLSVerifierCache(max_sets=blk, device=0) for _ in range(nctx)]
    bufs = [C.create_string_buffer(h_sets_bytes[(i * blk) * 320:((i + 1) * blk) * 320], blk * 320) for i in range(nctx)]
    oks = [0] * nctx

    def worker(i, count):
        good = 0
        for _ in range(count):
            good += 1 if L.blsgpu_batch_verify(caches[i].handle, bufs[i], blk, srb, chunks, None, None) == 1 else 0
        oks[i] = good

    def run(count):
        th = [threading.Thread(target=worker, args=(i, count)) for i in range(nctx)]
        t0 = time.perf_counter()
        for t in th:
            t.start()
        for t in th:
            t.join()
        return time.perf_counter() - t0

    run(2)                                                  # warm-up: programs compiled, buffers touched
    dt = run(batches_each)
    total = nctx * batches_each
    ok = sum(oks) == total
    for c in caches:
        c.close()
    return {"contexts": nctx, "batches": total, "batches_per_s": total / dt, "sets_per_s": total * blk / dt,
            "ms_per_batch_per_context": dt / batches_each * 1e3, "all_verified": ok}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--sets-per-gpu", type=int, default=SETS_PER_GPU)
    ap.add_argument("--chunks", type=int, default=-1, help="RLC chunk count (tp.numThreads); default: host hardware threads")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-msm", action="store_true", help="skip the G1 MSM extras")
    ap.add_argument("--no-msm-sweep", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="headline line only (profiling runs)")
    ap.add_argument("--msm-log2", type=int, default=20)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step returned (verdict, 576-byte GT, this "
                         "rank's 576-byte partial) to DIR/<name>.npy as float64, one value per byte, so that two builds "
                         "can be compared output for output; DIR/inputs.json records the seed and the RLC chunk count "
                         "(pin --chunks when the hosts differ)")
    args = ap.parse_args()
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist
    import nim_blscurve_b200 as bg

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    L = bg.lib()
    S = args.sets_per_gpu
    total = S * world
    chunks = args.chunks if args.chunks >= 0 else default_chunks(world)
    first = rank * S
    srb = hashlib.sha256(b"Mr F was here").digest()

    cache = bg.BatchedBLSVerifierCache(max_sets=S, device=local)
    h = cache.handle
    # ONE stream for everything in the timed region: torch's H2D copies, the library's kernels and the NCCL
    # all-gather are issued on it, so they are ordered without host synchronisation.  (torch's default stream has
    # handle 0, which blsgpu_set_stream reads as "use the context's own stream" - hence a dedicated stream.)
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    L.blsgpu_set_stream(h, C.c_void_p(stream.cuda_stream))

    # synthetic workload, generated on the device: rank r owns global sets [r*S, (r+1)*S)
    d_sets = torch.empty(S * 320, dtype=torch.uint8, device=dev)
    rc = L.blsgpu_make_sets(h, SEED, first, S, C.c_void_p(d_sets.data_ptr()), 1)
    assert rc == 0, cache.last_error()
    h_sets = torch.empty(S * 320, dtype=torch.uint8).pin_memory()
    h_sets.copy_(d_sets)
    d_partial = torch.zeros(576, dtype=torch.uint8, device=dev)
    d_all = torch.zeros(world * 576, dtype=torch.uint8, device=dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)      # > 126 MB L2
    gt = (C.c_uint8 * 576)()
    launches = [0]
    stage_acc = {}
    last_rc = [None]

    def step(src_ptr, n=S, first_=first, total_=total, chunks_=chunks, expect=1):
        # one collective: the 576-byte partial carries the share's verdict too (a flagged share seals it as zero)
        rc = L.blsgpu_partial_dev(h, C.c_void_p(src_ptr), n, first_, total_, srb, chunks_,
                                  C.c_void_p(d_partial.data_ptr()), None)
        assert rc == 0, cache.last_error()
        if world > 1:
            dist.all_gather_into_tensor(d_all, d_partial)
            rc = L.blsgpu_finalize_dev(h, C.c_void_p(d_all.data_ptr()), world, None, gt)
        else:
            rc = L.blsgpu_finalize_dev(h, C.c_void_p(d_partial.data_ptr()), 1, None, gt)
        launches[0] += L.blsgpu_last_launches(h)
        last_rc[0] = rc
        assert rc == expect, f"batch verdict {rc}, expected {expect}: {cache.last_error()}"
        ms = (C.c_float * 16)()
        k = L.blsgpu_last_stage_ms(h, ms, 16)
        for i in range(k):
            nm = L.blsgpu_stage_name(i).decode()
            stage_acc[nm] = stage_acc.get(nm, 0.0) + ms[i]

    def timed(fn, steps):
        """K steps bracketed by barrier + synchronize, device time by CUDA events, max over ranks."""
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(steps):
            flush.zero_()
            fn()
        e1.record(stream)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    def resident():
        step(d_sets.data_ptr())

    h_pageable = None
    if world == 1:
        h_pageable = bytearray(S * 320)                               # ordinary (pageable) host memory, like a Nim seq
        h_pageable[:] = h_sets.numpy().tobytes()
        c_pageable = (C.c_uint8 * (S * 320)).from_buffer(h_pageable)

    def e2e_plugin_pinned():
        rc = L.blsgpu_batch_verify(h, C.c_void_p(h_sets.data_ptr()), S, srb, chunks, None, gt)
        assert rc == 1, cache.last_error()

    def e2e_plugin_pageable():
        rc = L.blsgpu_batch_verify(h, c_pageable, S, srb, chunks, None, gt)
        assert rc == 1, cache.last_error()

    h_part = torch.zeros(576, dtype=torch.uint8).pin_memory()
    c_flag = C.c_int(0)

    def e2e_ranks():
        # the host-buffer share call of the ABI: H2D (overlapped with the hash inside the library), the share's pipeline,
        # its 576-byte partial back on the host; then the exchange and the one final exponentiation
        rc = L.blsgpu_partial(h, C.c_void_p(h_sets.data_ptr()), 0, S, first, total, srb, chunks, None,
                              C.c_void_p(h_part.data_ptr()), C.byref(c_flag))
        assert rc == 0, cache.last_error()
        d_partial.copy_(h_part, non_blocking=True)
        dist.all_gather_into_tensor(d_all, d_partial)
        rc = L.blsgpu_finalize_dev(h, C.c_void_p(d_all.data_ptr()), world, None, gt)
        assert rc == 1, cache.last_error()

    for _ in range(max(args.warmup, 3)):
        resident()
    stage_acc.clear()
    launches[0] = 0
    stop, samples = threading.Event(), []
    th = threading.Thread(target=clocks_sampler, args=(stop, samples, local), daemon=True)
    if rank == 0:
        th.start()
    ms_total = timed(resident, args.steps)
    stop.set()
    if args.dump_outputs and rank == 0:
        # the batch is the seeded device-generated workload, so with the same arguments and rlc_chunks these are
        # the same bytes on every run; the GT and the partial are copied before any later call overwrites them
        import numpy as np
        os.makedirs(args.dump_outputs, exist_ok=True)
        dumps = {"verdict": [last_rc[0]], "gt": bytes(gt), "partial": d_partial.cpu().numpy().tobytes()}
        for name, v in dumps.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), np.array(list(v), dtype=np.float64))
        # the GT and the partial depend on the RLC chunk count, which defaults to the host's thread count: pass --chunks
        # to compare dumps taken on different hosts
        with open(os.path.join(args.dump_outputs, "inputs.json"), "w") as f:
            json.dump({"seed": SEED, "sets_per_gpu": S, "world": world, "rlc_chunks": chunks, "srb": srb.hex()}, f)
    n_launch = launches[0]
    stages = {k: v / args.steps for k, v in stage_acc.items()}
    e2e_extra = {}
    if world == 1:
        for _ in range(2):
            e2e_plugin_pinned()
        ms_e2e = timed(e2e_plugin_pinned, args.steps)
        for _ in range(2):
            e2e_plugin_pageable()
        ms_pg = timed(e2e_plugin_pageable, args.steps)
        e2e_extra = {"call": "blsgpu_batch_verify(ctx, host sets, n, srb, chunks, NULL, gt) — the plugin entry, pinned host buffer",
                     "pageable": {"value": total * args.steps / (ms_pg * 1e-3), "unit": "sets/s", "ms_per_step": ms_pg / args.steps,
                                  "note": "same call from ordinary pageable host memory (a Nim seq)"}}
    else:
        for _ in range(2):
            e2e_ranks()
        ms_e2e = timed(e2e_ranks, args.steps)
        e2e_extra = {"call": "per rank: blsgpu_partial(pinned host share) -> 576-byte partial on the host -> NCCL all_gather(576 B) "
                             "-> blsgpu_finalize_dev"}
    value = total * args.steps / (ms_total * 1e-3)
    e2e_value = total * args.steps / (ms_e2e * 1e-3)

    # ---- parity inside the bench: the timed batch itself, corrupted, must be rejected with a GT that does not depend
    # on how the batch is cut (8 shares through a second context at N = 1; identical on every rank at N > 1) ----------
    parity = {}
    bad = d_sets.clone()
    victim = (S * 5) // 7
    bad[victim * 320 + 96 + 3] ^= 0x10                     # one message bit of one set of this rank's share
    step(bad.data_ptr(), expect=0)
    gt_bad = bytes(gt)
    parity["corrupted_batch_rejected"] = True
    if world == 1:
        c2 = bg.BatchedBLSVerifierCache(max_sets=S // 8 + 1, device=local)
        parts = b""
        for r in range(8):
            f8, n8 = bg.shard_range(S, 8, r)
            out = (C.c_uint8 * 576)()
            fl = C.c_int(0)
            rc = L.blsgpu_partial(c2.handle, C.c_void_p(bad.data_ptr() + f8 * 320), 1, n8, f8, S, srb, chunks, None, out, C.byref(fl))
            assert rc == 0 and fl.value == 0, c2.last_error()
            parts += bytes(out)
        g2 = (C.c_uint8 * 576)()
        rc = L.blsgpu_finalize(c2.handle, parts, 8, g2)
        assert rc == 0 and bytes(g2) == gt_bad, "GT of the corrupted timed batch differs between 1 and 8 shares"
        parity["gt_equals_8_share_gt_of_second_context"] = True
        c2.close()
    else:
        mine = torch.frombuffer(bytearray(gt_bad), dtype=torch.uint8).to(dev)
        allgt = torch.empty(world * 576, dtype=torch.uint8, device=dev)
        dist.all_gather_into_tensor(allgt, mine)
        allgt = allgt.cpu().numpy().tobytes()
        assert all(allgt[576 * r:576 * (r + 1)] == gt_bad for r in range(world)), "ranks disagree on the GT"
        parity["gt_identical_on_all_ranks"] = True
    del bad
    launches[0] = 0

    # ---- BASELINE configs[3]: ONE 32 768-set batch per step cut over the ranks (strong scaling of an epoch batch) ----
    extra = {}
    if not args.no_extras and S * world >= 32768 and 32768 % world == 0:
        S3 = 32768 // world

        def c3():
            step(d_sets.data_ptr(), n=S3, first_=rank * S3, total_=32768)
        # (the first S3 sets of every rank's share: distinct valid sets; the derivation is the global one of a 32 768 batch)
        for _ in range(3):
            c3()
        ms3 = timed(c3, args.steps)
        extra["config3"] = {"what": "BASELINE configs[3]: one 32768-set batch per step sharded over the ranks "
                                    "(blsgpu_partial_dev + one 576-byte all_gather + one final exponentiation)",
                            "sets": 32768, "sets_per_rank": S3, "ms_per_batch": ms3 / args.steps,
                            "sets_per_s": 32768 * args.steps / (ms3 * 1e-3), "rlc_chunks": chunks}

    if rank == 0:
        # roofline: integer-multiply pipe.  Peak = IMAD.WIDE multiply-accumulates/s measured by the microbenchmark
        # kernel in this same run; achieved = algorithmic Fp-mul of the dominant kernel x 300 / its event time.
        peak_wide = L.blsgpu_imad_peak(h, 1)
        peak_lo = L.blsgpu_imad_peak(h, 0)
        dom = max(STAGE_FPMUL, key=lambda k: stages.get(k, 0.0))
        dom_ms = stages[dom]
        achieved = S * STAGE_FPMUL[dom] * IMAD_PER_FPMUL / (dom_ms * 1e-3)
        whole = value / world * (W_SET * IMAD_PER_FPMUL)
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        hbm_peak = peaks.get("hbm_gbs", 6650.0)
        traffic, traffic_src = ncu_traffic(STAGE_KERNEL.get(dom, dom))
        executed = EXECUTED_IMAD_WIDE_PER_SET.get(dom)
        extra["roofline"] = {
            "bound": "int_mul_pipe", "kernel": dom, "achieved": achieved / 1e9, "peak": peak_wide / 1e9,
            "unit": "G IMAD.WIDE/s", "frac": achieved / peak_wide,
            "frac_note": "reference-algorithm work (SURVEY.md §8a Fp-mul counts x 300) / kernel time / measured peak",
            "frac_executed": (S * executed / (dom_ms * 1e-3) / peak_wide) if executed else None,
            "frac_executed_note": "IMAD.WIDE lane-operations the kernel actually executes per set (ncu source page of the "
                                  "committed capture) / kernel time / the same peak: the kernel does less work than the "
                                  "reference algorithm (dedicated squaring, two-chain square root)",
            "traffic": traffic,
            "traffic_note": "DRAM bytes read+written per launch of %s, ncu --set full on the same 131072-set workload (%s); "
                            "algorithmic bytes per launch are %d (inputs + outputs) - the rest is per-thread stack "
                            "(local memory) traffic that overflows L2" % (STAGE_KERNEL.get(dom, dom), traffic_src,
                                                                          S * STAGE_IO_BYTES.get(dom, 320)),
            "kernel_ms": dom_ms, "algorithmic_fpmul_per_set": STAGE_FPMUL[dom], "imad_per_fpmul": IMAD_PER_FPMUL,
            "peak_source": "k_imad_peak microbenchmark in this run (mad.wide.u32; not in MEASURED_PEAKS.json, which holds "
                           "HBM and bf16 only); mad.lo.u32 peak %.1f G/s; a-priori bound of SURVEY.md §8d 18600 G/s" % (peak_lo / 1e9),
            "frac_of_apriori_bound": achieved / 1.86e13,
            "whole_step_frac": whole / peak_wide,
            "hbm": {"achieved_gbs": S * 320 / (ms_total / args.steps * 1e-3) / 1e9, "peak_gbs": hbm_peak,
                    "note": "320 B of input per set: HBM is not the bound (%s)" %
                            ("of measured" if "hbm_gbs" in peaks else "of fallback")},
        }
        extra["stages_ms"] = stages
        extra["parity_checks"] = parity
        br = None
        cores = host_threads()
        if not args.no_cpu_baseline:
            try:
                from oracle import blst_ref as br
                cores = br.ncores()
            except Exception:
                br = None
        sets_host = h_sets.numpy().tobytes()[:max(4096, 129 * 40) * 320] if not args.no_extras else b""

        def wall(fn, reps, warm=3):
            for _ in range(warm):
                fn()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(reps):
                r = fn()
            return (time.perf_counter() - t0) / reps, r

        if not args.no_extras:
            # ---- BASELINE configs[0]: 64 distinct-message sets, serial and 4-chunk derivation, host call ----
            c64 = (C.c_uint8 * (64 * 320)).from_buffer_copy(sets_host[:64 * 320])
            cfg1 = {"what": "BASELINE configs[0]: batchVerify of 64 distinct-message sets, blsgpu_batch_verify from a host "
                            "buffer, wall clock per call (latency-bound)", "sets": 64}
            for ch in (0, 4):
                t, r = wall(lambda: L.blsgpu_batch_verify(h, c64, 64, srb, ch, None, gt), 10)
                cfg1["chunks_%d" % ch] = {"ms": t * 1e3, "sets_per_s": 64 / t, "verified": r == 1}
            if br is not None:
                t16 = br.time_batch_verify(sets_host[:64 * 320], srb, cores, 5)
                t1 = br.time_batch_verify(sets_host[:64 * 320], srb, 1, 2)
                cfg1["cpu_baseline"] = {"value": t16 * 1e3, "unit": "ms", "cores": cores, "kind": "reference",
                                        "sample": f"the same 64 sets, BLST batchVerifyParallel replica, {cores} threads, best of 5; "
                                                  f"batchVerifySerial on one thread: {t1 * 1e3:.1f} ms"}
            extra["config1"] = cfg1
            # ---- Eth2 block batch (configs[1]): 129 sets, latency-bound ----
            blk = 129
            tb, rcb = wall(lambda: L.blsgpu_batch_verify_dev(h, C.c_void_p(d_sets.data_ptr()), blk, srb, 4, None, gt), 5)
            extra["block_batch"] = {"sets": blk, "ms": tb * 1e3, "sets_per_s": blk / tb, "verified": rcb == 1,
                                    "what": "BASELINE configs[1]: 129-set batch (128 attestations + 1 sync committee), host call "
                                            "blsgpu_batch_verify_dev, wall clock; latency-bound"}
            cblk = (C.c_uint8 * (blk * 320)).from_buffer_copy(sets_host[:blk * 320])
            tbh, rch = wall(lambda: L.blsgpu_batch_verify(h, cblk, blk, srb, 4, None, gt), 5)
            extra["block_batch"]["ms_from_host_buffer"] = tbh * 1e3
            # stage breakdown: event timing does not exist inside a replayed CUDA graph, so a second context with graphs off
            os.environ["BLSGPU_GRAPH"] = "0"
            c_ng = bg.BatchedBLSVerifierCache(max_sets=blk, device=local)
            del os.environ["BLSGPU_GRAPH"]
            tng, _ = wall(lambda: L.blsgpu_batch_verify(c_ng.handle, cblk, blk, srb, 4, None, gt), 5)
            ms_ = (C.c_float * 16)()
            kk = L.blsgpu_last_stage_ms(c_ng.handle, ms_, 16)
            extra["block_batch"]["stages_ms"] = {L.blsgpu_stage_name(i).decode(): ms_[i] for i in range(kk)}
            extra["block_batch"]["ms_without_cuda_graph"] = tng * 1e3
            extra["block_batch"]["launches_without_cuda_graph"] = L.blsgpu_last_launches(c_ng.handle)
            c_ng.close()
            # the same block with the public-key aggregation done on the GPU first: 128 committees x 128 keys + one of 512
            nkeys = min(128 * 128 + 512, (S // 129) * 129)
            member = bytes(h_sets[:nkeys * 320].numpy().reshape(nkeys, 320)[:, :96].tobytes())
            offs = [min(128 * i, nkeys) for i in range(129)] + [nkeys]
            c_offs = (C.c_uint32 * len(offs))(*offs)
            agg_out = (C.c_uint8 * (96 * 129))()
            ta, rca = wall(lambda: L.blsgpu_aggregate_g1_segments(h, member, c_offs, 129, agg_out), 5, warm=2)
            extra["block_batch"].update({"key_aggregation_ms": ta * 1e3, "keys_aggregated": nkeys, "aggregation_ok": rca == 1,
                                         "ms_with_key_aggregation": (tb + ta) * 1e3})
            # single pairing checks through the verify entry points (timing only: the signature is another set's)
            pk512 = member[:512 * 96]
            sig = sets_host[128:320]
            msg = sets_host[96:128]
            dst = bg.batch_verifier.DST
            tf, _ = wall(lambda: L.blsgpu_fast_aggregate_verify(h, pk512, 512, msg, 32, dst, len(dst), sig, None), 5)
            offs2 = (C.c_uint32 * 2)(0, 32)
            tv, rv = wall(lambda: L.blsgpu_aggregate_verify(h, sets_host[:96], 1, msg, offs2, dst, len(dst), sig, None), 5)
            extra["verify_entry_points"] = {"fast_aggregate_verify_512_keys_ms": tf * 1e3, "verify_ms": tv * 1e3,
                                            "verify_ok": rv == 1,
                                            "what": "one pairing check per call (bls_sig_min_pubkey.nim:108-258), host buffers, wall clock"}
            # ---- batch-size sweep (sets resident, wall clock per call, chunks as the headline) ----
            sweep = {}
            for n_ in (256, 1024, 2048, 4096, 8192, 16384, 32768, 65536):
                if n_ > S:
                    break
                t, r = wall(lambda: L.blsgpu_batch_verify_dev(h, C.c_void_p(d_sets.data_ptr()), n_, srb, chunks, None, gt), 3, warm=2)
                sweep[str(n_)] = {"ms": t * 1e3, "sets_per_s": n_ / t, "verified": r == 1}
            extra["batch_sizes"] = sweep
            # ---- the same 131072-set step under other RLC chunk counts (sequential SHA-256 chains of n/chunks) ----
            cs = {}
            for ch in (0, 16, 64, 1024):
                t, r = wall(lambda: L.blsgpu_batch_verify_dev(h, C.c_void_p(d_sets.data_ptr()), S, srb, ch, None, gt), 2, warm=1)
                cs[str(ch)] = {"ms": t * 1e3, "sets_per_s": S / t, "verified": r == 1}
            extra["chunk_sweep"] = {"sets": S, "by_rlc_chunks": cs,
                                    "note": "chunks = 0 is batchVerifySerial's single chain of n SHA-256 blocks; batchVerify picks the "
                                            "parallel derivation whenever tp.numThreads > 1 (bls_batch_verifier.nim:440)"}
            # ---- streaming blocks: K contexts in flight, 129-set batches from host buffers ----
            if world == 1:
                torch.cuda.synchronize()
                sb = {}
                for k_ in (1, 8, 32):
                    sb["contexts_%d" % k_] = bench_streaming(L, bg, sets_host, srb, blk, k_, 24 if k_ > 1 else 40, 4)
                best = max(sb.values(), key=lambda v: v["batches_per_s"])
                extra["streaming_blocks"] = {"what": "K host threads, one context each on ONE GPU, back-to-back blsgpu_batch_verify of "
                                                     "129-set batches from host buffers (wall clock)", "runs": sb,
                                             "batches_per_s": best["batches_per_s"], "sets_per_s": best["sets_per_s"]}
            if not args.no_msm:
                extra["msm_g1"] = bench_msm(L, h, stream, flush, peak_wide, hbm_peak, args)
        if world == 1 and br is not None:
            n = max(64, min(S, 2500 * cores))
            sample = h_sets[:n * 320].numpy().tobytes()
            t = br.time_batch_verify(sample, srb, cores, 1)
            t1n = min(n, 4096)
            t1 = br.time_batch_verify(sample[:t1n * 320], srb, 1, 1)
            extra["cpu_baseline"] = {
                "value": n / t, "unit": "sets/s", "cores": cores, "kind": "reference",
                "sample": f"first {n} sets of the same workload, BLST (oracle/_ref) batchVerifyParallel replica, "
                          f"{cores} threads, one run; single-thread: {t1n / t1:.0f} sets/s on {t1n} sets"}
            if "block_batch" in extra:
                # the 129-set block batch on the host cores as well (best of 5: it is a latency comparison)
                tblk = br.time_batch_verify(sample[:129 * 320], srb, cores, 5)
                extra["block_batch"]["cpu_baseline"] = {
                    "value": tblk * 1e3, "unit": "ms", "cores": cores, "kind": "reference",
                    "sample": f"the same 129 sets, BLST batchVerifyParallel replica, {cores} threads, best of 5"}
                if "streaming_blocks" in extra:
                    extra["streaming_blocks"]["cpu_baseline"] = {
                        "value": 1.0 / tblk, "unit": "batches/s", "cores": cores, "kind": "reference",
                        "sample": f"back-to-back BLST batchVerifyParallel of the same 129 sets on {cores} threads (1 / best-of-5 latency)"}
                    extra["streaming_blocks"]["vs_cpu"] = extra["streaming_blocks"]["batches_per_s"] * tblk
        elif world == 1 and not args.no_cpu_baseline:
            extra["cpu_baseline"] = {"value": None, "unit": "sets/s", "cores": 0, "kind": "reference", "sample": "oracle unavailable"}
        cfg = make_config(S, world, chunks)
        line = {
            "metric": "batch-verified signature sets/sec", "value": value, "unit": "sets/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_total / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u32x12 (Fp 381-bit Montgomery)", "data": "synthetic",
            "config": cfg,
            "clocks": summarize_clocks(samples),
            "e2e": dict({"value": e2e_value, "unit": "sets/s", "h2d_bytes_per_step": S * 320 * world,
                         "d2h_bytes_per_step": (576 + 16) * world, "ms_per_step": ms_e2e / args.steps}, **e2e_extra),
            "gpu_launches": n_launch,
        }
        line.update(extra)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
