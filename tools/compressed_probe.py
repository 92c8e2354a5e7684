"""Time batch verification of compressed signature sets against the two ways a caller can do without it.

  (a) blsgpu_batch_verify on 320-byte sets (signatures already decoded)
  (b) blsgpu_batch_verify_compressed on 224-byte sets (decode + subgroup check inside the pipeline)
  (c) blsgpu_signatures_from_bytes (decode + subgroup check), a host repack into 320-byte sets, blsgpu_batch_verify

Host buffers, host wall clock around each call (every call ends with a device synchronise), arms warmed up and then
alternated.  The card name and power limit are read in the same run.  Usage:
  python tools/compressed_probe.py [--sizes 129,4096,32768,131072] [--reps 7] [--out FILE]
The rows are printed as they are measured; --out also writes the whole result as one JSON file.
"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import nim_blscurve_b200 as bg  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="129,4096,32768,131072")
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--chunks", type=int, default=16)
    ap.add_argument("--out", default=None, help="write the whole result to this JSON file")
    a = ap.parse_args()
    sizes = [int(x) for x in a.sizes.split(",")]
    L = bg.lib()
    cache = bg.BatchedBLSVerifierCache(max_sets=max(sizes), device=0)
    h = cache.handle
    srb = bytes(range(32))
    rows = []
    for n in sizes:
        buf = (C.c_uint8 * (320 * n))()
        assert L.blsgpu_make_sets(h, 1234 + n, 0, n, buf, 0) == 0
        sets = np.frombuffer(bytes(buf), dtype=np.uint8).reshape(n, 320)
        comp = np.frombuffer(bg.signaturesToBytes(cache, sets[:, 128:].tobytes()), dtype=np.uint8).reshape(n, 96)
        sets320 = sets.tobytes()
        sets224 = np.concatenate([sets[:, :128], comp], axis=1).tobytes()
        comp96 = comp.tobytes()
        status = (C.c_uint8 * n)()
        dec = (C.c_uint8 * (192 * n))()

        def arm_a():
            return L.blsgpu_batch_verify(h, sets320, n, srb, a.chunks, None, None)

        def arm_b():
            return L.blsgpu_batch_verify_compressed(h, sets224, n, srb, a.chunks, None, None, status)

        def arm_c():
            ok = L.blsgpu_signatures_from_bytes(h, comp96, n, 96, 1, dec, status)
            if ok != 1:
                return 0 if ok == 0 else ok
            d = np.frombuffer(dec, dtype=np.uint8).reshape(n, 192)
            repacked = np.concatenate([sets[:, :128], d], axis=1).tobytes()
            return L.blsgpu_batch_verify(h, repacked, n, srb, a.chunks, None, None)

        arms = {"a_sets320": arm_a, "b_compressed": arm_b, "c_from_bytes_repack": arm_c}
        verdicts = {k: set() for k in arms}
        for _ in range(3):                                   # warm-up: modules, programs, graphs, staging
            for k, f in arms.items():
                verdicts[k].add(f())
        times = {k: [] for k in arms}
        for _ in range(a.reps):
            for k, f in arms.items():
                t0 = time.perf_counter()
                rc = f()
                times[k].append((time.perf_counter() - t0) * 1e3)
                verdicts[k].add(rc)
        assert all(v == {1} for v in verdicts.values()), verdicts
        med = {k: statistics.median(v) for k, v in times.items()}
        row = {"n": n, "median_ms": {k: round(v, 3) for k, v in med.items()},
               "min_ms": {k: round(min(v), 3) for k, v in times.items()},
               "b_minus_a_ms": round(med["b_compressed"] - med["a_sets320"], 3),
               "b_over_a": round(med["b_compressed"] / med["a_sets320"], 4),
               "b_faster_than_c": med["b_compressed"] < med["c_from_bytes_repack"], "verdicts_agree": True}
        print(json.dumps(row), flush=True)
        rows.append(row)
    out = {"card": card(), "chunks": a.chunks, "reps": a.reps,
           "method": "host buffers; host wall clock per call (each call ends with a device synchronise); 3 warm-up rounds, "
                     "then the three arms alternated; median and minimum over the reps",
           "rows": rows}
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(out, f, indent=1)
    print(json.dumps({"card": out["card"]}))
    cache.close()


if __name__ == "__main__":
    main()
