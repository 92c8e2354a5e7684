"""Every batch route on degenerate signature sets, verdict and all 576 GT bytes against a pyref reference.

The batch pipeline picks its kernels by batch size (route.hpp), and each route has its own code for the cases that make
a batch degenerate: a signature sum S = sum r_i sig_i at infinity (the neutral lines of k_lines_from_prog, the infinity
test of k_miller_lines_lanes2 and miller_lines, pt_to_affine_vt in k_sig_pair, the deferred one-pair loop on ml_sig),
infinite public keys (the flag k_g1_mul raises, cleared at the start of every call), repeated points with equal scalars
(P + P and P - P in the G2 tree and the Pippenger buckets), and the final exponentiation of arbitrary partials.

The sizes come from route.hpp through hostsim: the first and the last batch size of every run of equal plans, so a
moved threshold moves the sizes.  The reference is pyref by bilinearity: the sets are built from a small pool of
points, so the expected GT is one final exponentiation of at most four Miller loops whatever the batch size.  A CPU test
checks that reference against pyref.batch_verify set by set on small batches of every scenario."""
import ctypes as C
import functools
import hashlib
import json
import os
import random
import subprocess
import sys

import numpy as np
import pytest

from oracle import pyref as pr

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
Q = pr.R_ORDER
ONE_GT = pr.f12_to_bytes(pr.F12_ONE)
ZERO_GT = bytes(576)
ERR_ARG = -2                                     # include/blsgpu.h
gpu = pytest.mark.gpu


# ---- sizes from route.hpp ------------------------------------------------------------------------------------------
@functools.lru_cache(maxsize=None)
def _hostsim():
    so = os.path.join(HERE, "hostsim", "libhostsim.so")
    src = os.path.join(HERE, "hostsim", "hostsim.cpp")
    csrc = os.path.join(ROOT, "nim_blscurve_b200", "csrc")
    deps = [src] + [os.path.join(csrc, f) for f in os.listdir(csrc) if f.endswith((".cuh", ".hpp"))]
    if not os.path.exists(so) or any(os.path.getmtime(d) > os.path.getmtime(so) for d in deps):
        subprocess.run(["g++", "-O2", "-shared", "-fPIC", "-x", "c++", "-std=c++17", "-o", so, src], check=True)
    return C.CDLL(so)


N_MAX = 40000
# hostsim.cpp hs_plan_routes: the batch plan, then the lines route of the Miller plan of the pairs the batch runs
PLAN_FIELDS = ["hash", "sliced", "small", "sig", "g1_aside", "msm_after_hash", "defer_sig", "affine", "chain_hog",
               "chain_wait", "graph", "copy_ahead", "lines", "lines_last"]
# (chunks, host source, explicit scalars)
CONFIGS = [(chunks, host, scalars) for chunks in (0, 64) for host in (1, 0) for scalars in (0, 1)]
# sizes no plan marks: the first levels of the pairwise G2 tree, and both sides of the 128 sets of one block of the
# per-set kernels (k_g1_mul stages 128 sets per block)
TREE_AND_BLOCK_EDGES = (2, 3, 127, 128, 129)


@functools.lru_cache(maxsize=None)
def route_table(chunks, host, scalars):
    """plans of the batches of 1 .. N_MAX sets: N_MAX x 14 ints, row n - 1 for n sets"""
    out = np.zeros(N_MAX * len(PLAN_FIELDS), dtype=np.int32)
    _hostsim().hs_plan_routes(C.c_size_t(N_MAX), C.c_uint32(chunks), host, scalars, out.ctypes.data_as(C.c_void_p))
    return out.reshape(N_MAX, len(PLAN_FIELDS))


def plan_runs(table):
    """[(first n, last n)] of every run of equal plans"""
    cut = np.nonzero(np.any(table[1:] != table[:-1], axis=1))[0] + 1      # row index where a new run starts
    starts = [0] + [int(c) for c in cut]
    ends = [s - 1 for s in starts[1:]] + [len(table) - 1]
    return [(s + 1, e + 1) for s, e in zip(starts, ends)]


@functools.lru_cache(maxsize=None)
def route_sizes():
    sizes = set(TREE_AND_BLOCK_EDGES)
    for cfg in CONFIGS:
        for first, last in plan_runs(route_table(*cfg)):
            sizes.update((first, last))
    return sorted(sizes)


SIZES = route_sizes()


# ---- the pool and the scenarios ------------------------------------------------------------------------------------
# A set is (a, k, sig): public key [a]G1 (a None: infinity), message MSGS[k], signature [b]B for sig = (B, b) with B a
# message index (B = H(MSGS[B])) or "X" (a fixed G2 point), or None (infinity).  Scalars are kept mod q.
MSGS = [hashlib.sha256(b"degenerate batches %d" % k).digest() for k in range(3)]
KEYS = [random.Random(2026).getrandbits(64) | 1 for _ in range(16)]
TABLE = [3, 5, 7, 11, 13]                        # the free coefficients of the scenarios that solve for the last one


@functools.lru_cache(maxsize=None)
def _hash(k):
    return pr.hash_to_g2(MSGS[k])


def _base(b):
    return pr.G2_GEN if b == "X" else _hash(b)


@functools.lru_cache(maxsize=None)
def _pk(a):
    return None if a is None else pr.g1_mul(pr.G1_GEN, a)


@functools.lru_cache(maxsize=None)
def _sig(sig):
    return None if sig is None else pr.g2_mul(_base(sig[0]), sig[1])


@functools.lru_cache(maxsize=None)
def _set_bytes(s):
    a, k, sig = s
    return pr.g1_to_mem(_pk(a)) + MSGS[k] + pr.g2_to_mem(_sig(sig))


def encode(batch):
    return b"".join(_set_bytes(s) for s in batch)


def valid_set(i):
    j = i % len(KEYS)
    return (KEYS[j], j % 3, (j % 3, KEYS[j]))


def valid(n):
    return [valid_set(i) for i in range(n)]


def edge_positions(n, rng=None):
    """0, n - 1, both sides of the first 128-set block, n / 2, and about 1 % of the sets at random"""
    pos = {p for p in (0, n - 1, 127, 128, n // 2) if p < n}
    if rng is not None:
        pos.update(rng.sample(range(n), n // 100))
    return sorted(pos)


def solve_last(r, coeffs):
    """the last coefficient c such that sum r_i c_i == 0 (mod q), the others given"""
    s = sum(ri * ci for ri, ci in zip(r, coeffs)) % Q
    return -s * pow(r[len(coeffs)], -1, Q) % Q


def infinite_signatures(n):
    b = valid(n)
    for p in edge_positions(n, random.Random(n)):
        b[p] = b[p][:2] + (None,)
    return b


def all_signatures_infinite(n):
    return [s[:2] + (None,) for s in valid(n)]


def signature_sum_cancels(n, r):
    """sig_i = [c_i]X with sum r_i c_i == 0: S is infinity while signatures were aggregated; valid keys"""
    cs = [TABLE[i % len(TABLE)] for i in range(n - 1)]
    cs.append(solve_last(r, cs))
    return [s[:2] + ((("X", c) if c else None),) for s, c in zip(valid(n), cs)]


def accepting_at_infinity(n, r):
    """one message, pk_i = [a_i]G1, sig_i = [a_i]H with sum r_i a_i == 0: both sides of the check are at infinity, the
    verdict is true and the GT one (n >= 2)"""
    a = [TABLE[i % len(TABLE)] for i in range(n - 1)]
    a.append(solve_last(r, a))
    assert a[-1] != 0
    return [(x, 0, (0, x)) for x in a]


def infinite_keys(n):
    b = valid(n)
    for p in (0, n - 1, 127, 128):
        if p < n:
            b[p] = (None,) + b[p][1:]
    return b


def repeated(n):
    return [valid_set(0)] * n


def plus_minus(n):
    """(pk, m, sig), (-pk, m, -sig), ...: under equal scalars both sums are at infinity (odd n: one more valid set)"""
    a, k, _ = valid_set(0)
    pair = [(a, k, (k, a)), (Q - a, k, (k, Q - a))]
    return (pair * (n // 2) + [valid_set(0)] * (n % 2))[:n]


def reference(batch, r):
    """(verdict, GT bytes) of the batch under scalars r by bilinearity:
    GT = FE( conj(ML(G1, S)) * prod_k ML([c_k]G1, H_k) ),  c_k = sum of r_i a_i over the sets on message k,
    S = sum over the signature bases B of [sum r_i b_i]B.  An infinite public key gives (False, 576 zero bytes)."""
    if any(a is None for a, _, _ in batch):
        return False, ZERO_GT
    c, s = {}, {}
    for (a, k, sig), ri in zip(batch, r):
        c[k] = (c.get(k, 0) + ri * a) % Q
        if sig is not None:
            s[sig[0]] = (s.get(sig[0], 0) + ri * sig[1]) % Q
    f = pr.F12_ONE
    for k, ck in sorted(c.items()):
        if ck:
            f = pr.f12_mul(f, pr.miller_loop(pr.g1_mul(pr.G1_GEN, ck), _hash(k)))
    S = None
    for b, sb in sorted(s.items(), key=lambda x: str(x[0])):
        if sb:
            S = pr.g2_add(S, pr.g2_mul(_base(b), sb))
    if S is not None:
        f = pr.f12_mul(f, pr.f12_conj(pr.miller_loop(pr.G1_GEN, S)))
    out = pr.final_exp(f)
    return out == pr.F12_ONE, pr.f12_to_bytes(out)


@functools.lru_cache(maxsize=2)
def scenarios(n, srb):
    """(name, batch, scalars, chunks, explicit) of every scenario at size n"""
    r0, r64 = pr.rlc_scalars(srb, n, 0), pr.rlc_scalars(srb, n, 64)
    rx = [random.Random(n + 7).getrandbits(64) | 1 for _ in range(n)]
    out = [("infinite_signatures", infinite_signatures(n), r64, 64, False),
           ("all_signatures_infinite", all_signatures_infinite(n), r0, 0, False),
           ("signature_sum_cancels", signature_sum_cancels(n, r0), r0, 0, False),
           ("signature_sum_cancels_explicit", signature_sum_cancels(n, rx), rx, 0, True),
           ("infinite_keys", infinite_keys(n), r0, 0, False),
           ("repeated", repeated(n), r64, 64, False),
           ("repeated_ones", repeated(n), [1] * n, 0, True),
           ("repeated_max", repeated(n), [2 ** 64 - 1] * n, 0, True),
           ("plus_minus_max", plus_minus(n), [2 ** 64 - 1] * n, 0, True)]
    if n >= 2:
        out += [("accepting_at_infinity", accepting_at_infinity(n, r0), r0, 0, False),
                ("accepting_at_infinity_explicit", accepting_at_infinity(n, rx), rx, 0, True)]
    return out


# ---- CPU: the reference, the sizes, the final-exponentiation programs ----------------------------------------------
@pytest.mark.parametrize("n", [1, 3, 8])
def test_reference_against_pyref_batch_verify(srb, n):
    """The bilinear reference equals pyref.batch_verify run set by set, on every scenario; the solved scenarios do sum
    to zero and the accepting ones accept."""
    for name, batch, r, chunks, explicit in scenarios(n, srb):
        sets = [(_pk(a), MSGS[k], _sig(sig)) for a, k, sig in batch]
        ok, gt = pr.batch_verify(sets, srb, chunks, r if explicit else None)
        assert reference(batch, r) == (ok, gt if gt is not None else ZERO_GT), name
        if name.startswith("signature_sum_cancels"):
            S = None
            for (_, _, sig), ri in zip(sets, r):
                S = pr.g2_add(S, pr.g2_mul(sig, ri) if sig is not None else None)
            assert S is None and (n == 1 or all(s[2] is not None for s in sets)), name
        if name.startswith(("accepting", "repeated", "plus_minus")):
            assert (ok, gt) == (True, ONE_GT), name
        assert [pr.g1_from_mem(raw[:96]) for raw in map(_set_bytes, batch)] == [s[0] for s in sets]


def test_route_sizes_reach_every_plan():
    """The GPU tests run the first and the last size of every run of equal plans (batch plan + the lines route of the
    Miller plan the batch runs) under derived and explicit scalars, from host and device memory, in 0 and 64 chunks:
    every plan that occurs for 1 .. N_MAX sets occurs at one of those sizes."""
    seen = set()
    for cfg in CONFIGS:
        t = route_table(*cfg)
        every = {tuple(row) for row in t.tolist()}
        at_sizes = {tuple(t[n - 1].tolist()) for n in SIZES}
        assert every == at_sizes, cfg
        seen |= {(cfg,) + p for p in every}
    assert SIZES[0] == 1 and SIZES[-1] == N_MAX
    # the boundaries the routes are known to have (route.hpp read_thresholds) are among them
    for n in (1024, 1025, 2048, 2049, 2499, 2500, 4096, 4097, 4499, 4500, 8192, 8193, 32767, 32768, 35999, 36000):
        assert n in SIZES, n
    print(f"{len(seen)} distinct (configuration, plan) pairs, "
          f"{len({p[1:] for p in seen})} distinct plans; sizes {SIZES}")


FINAL_DIRECT_MAX = 8                             # blsgpu.cu: more partials are folded by product programs first


def test_final_programs_fit_for_the_partials_they_take():
    """fpprog::build_final reserves 12 slots per partial from the first round on: the pair of programs the device runs
    builds for 1 .. FINAL_DIRECT_MAX partials, and stops fitting the slot file long before 64 — so the library folds
    larger counts with product programs before the final exponentiation."""
    hs = _hostsim()
    builds = [c for c in range(1, 70) if hs.hs_prog_final_builds(c)]
    assert builds == list(range(1, builds[-1] + 1))
    assert FINAL_DIRECT_MAX <= builds[-1] < 64, builds[-1]
    print(f"largest count for which build_final builds: {builds[-1]}")


# ---- GPU -----------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module", params=SIZES, ids=lambda n: "n%d" % n)
def sized(request):
    import nim_blscurve_b200 as bg
    c = bg.BatchedBLSVerifierCache(max_sets=request.param, device=0)
    yield request.param, c
    c.close()


def _run(cache, batch, srb, chunks, r, explicit):
    return cache.verify_raw(encode(batch), srb, chunks, scalars=r if explicit else None, want_gt=True)


@gpu
def test_rlc_scalars_per_size(sized, srb):
    import nim_blscurve_b200 as bg
    n, c = sized
    for chunks in (0, 64):
        assert bg.rlcScalars(c, srb, n, chunks) == pr.rlc_scalars(srb, n, chunks), chunks


@gpu
def test_infinite_signatures(sized, srb):
    """infinite signatures at the edges and at random, then every signature infinite (S infinite, nothing aggregated)"""
    n, c = sized
    for name, batch, r, chunks, explicit in scenarios(n, srb)[:2]:
        want = reference(batch, r)
        assert want[0] is False
        assert _run(c, batch, srb, chunks, r, explicit) == want, name


@gpu
def test_signature_sum_cancels(sized, srb):
    """signatures [c_i]X with sum r_i c_i == 0 (mod q): S is infinity on every route that sums the signatures (per-set
    programs and tree, k_g2_mul and tree, Pippenger; the deferred pair and graph replay under derived scalars)"""
    n, c = sized
    for name, batch, r, chunks, explicit in scenarios(n, srb)[2:4]:
        want = reference(batch, r)
        assert want[0] is False
        assert _run(c, batch, srb, chunks, r, explicit) == want, name


@gpu
def test_accepting_batch_with_signature_sum_at_infinity(sized, srb):
    """both sums at infinity: a wrong neutral line for the signature pair changes the GT from one"""
    n, c = sized
    if n < 2:
        pytest.skip("one set cannot cancel")
    for name, batch, r, chunks, explicit in scenarios(n, srb)[9:]:
        assert _run(c, batch, srb, chunks, r, explicit) == (True, ONE_GT), name


@gpu
def test_infinite_public_keys(sized, srb):
    n, c = sized
    name, batch, r, chunks, explicit = scenarios(n, srb)[4]
    assert _run(c, batch, srb, chunks, r, explicit) == (False, ZERO_GT)
    rx = [random.Random(n).getrandbits(64) | 1 for _ in range(n)]
    assert _run(c, batch, srb, 0, rx, True) == (False, ZERO_GT)


@gpu
def test_one_set_repeated(sized, srb):
    """one set n times under derived and equal explicit scalars (P + P in the trees and buckets), and (pk, m, sig) /
    (-pk, m, -sig) pairs under equal scalars (P - P); an explicit zero scalar is an argument error"""
    import nim_blscurve_b200 as bg
    n, c = sized
    for name, batch, r, chunks, explicit in scenarios(n, srb)[5:9]:
        assert _run(c, batch, srb, chunks, r, explicit) == (True, ONE_GT), name
    assert _run(c, plus_minus(n), srb, 0, [1] * n, True) == (True, ONE_GT)
    sc = (C.c_uint64 * n)(*([5] * n))
    sc[n // 2] = 0
    gt = (C.c_uint8 * 576)()
    assert bg.lib().blsgpu_batch_verify(c.handle, encode(repeated(n)), n, srb, 0, sc, gt) == ERR_ARG
    assert bytes(gt) == ZERO_GT


def _call_sequence(n):
    """valid -> infinite key -> valid -> S cancels -> valid -> accepting at infinity, each under its own random bytes"""
    seq = []
    for k, kind in enumerate(["valid", "keys", "valid", "cancels", "valid", "accepting"]):
        srb = hashlib.sha256(b"call order %d %d" % (n, k)).digest()
        r = pr.rlc_scalars(srb, n, 0)
        if kind == "valid":
            batch, want = valid(n), (True, ONE_GT)
        elif kind == "keys":
            batch, want = infinite_keys(n), (False, ZERO_GT)
        elif kind == "cancels":
            batch = signature_sum_cancels(n, r)
            want = reference(batch, r)
        else:
            if n < 2:
                continue
            batch, want = accepting_at_infinity(n, r), (True, ONE_GT)
        seq.append((kind, encode(batch), srb, want))
    return seq


@gpu
def test_call_order_on_one_context(sized):
    """One context, host and then device batches: each call gives what a fresh context gives, after an infinite key
    and whatever preceded it.  Up to 8 192 sets the third call with the same buffer and size replays a captured graph,
    with new random bytes each time."""
    import torch
    import nim_blscurve_b200 as bg
    n, c = sized
    seq = _call_sequence(n)
    for kind, raw, srb, want in seq:
        assert c.verify_raw(raw, srb, 0, want_gt=True) == want, ("host", kind)
    L = bg.lib()
    d = torch.empty(320 * n, dtype=torch.uint8, device="cuda")
    gt = (C.c_uint8 * 576)()
    for kind, raw, srb, want in seq:
        d.copy_(torch.frombuffer(bytearray(raw), dtype=torch.uint8))
        torch.cuda.synchronize()
        rc = L.blsgpu_batch_verify_dev(c.handle, C.c_void_p(d.data_ptr()), n, srb, 0, None, gt)
        assert rc >= 0, c.last_error()
        assert (bool(rc), bytes(gt)) == want, ("device", kind)


_CHILD = r'''
import json, sys
sys.path.insert(0, sys.argv[1])
import nim_blscurve_b200 as bg
jobs = json.load(open(sys.argv[2]))
c = bg.BatchedBLSVerifierCache(max_sets=jobs["n"], device=0)
out = []
for j in jobs["calls"]:
    raw = open(j["path"], "rb").read()
    ok, gt = c.verify_raw(raw, bytes.fromhex(j["srb"]), j["chunks"], scalars=j["scalars"], want_gt=True)
    out.append([ok, gt.hex()])
c.close()
print(json.dumps(out))
'''


@gpu
@pytest.mark.parametrize("env", [{"BLSGPU_PAIR_HASH_MAX": "1", "BLSGPU_PAIR_LINES_MAX": "1"}, {"BLSGPU_SERIAL_TAIL": "1"}],
                         ids=["thread_per_set", "serial_tail"])
def test_degenerate_batches_in_a_child_process(tmp_path, srb, env):
    """The thread-per-set hash and lines kernels (default only beyond 125 000 / 180 000 sets) and the serial tail
    (single-thread final exponentiation and combine, no per-set programs, no graph), on a mid-size batch of every
    scenario, in a child process with the thresholds overridden."""
    n = 9000
    calls, wants = [], []
    for name, batch, r, chunks, explicit in scenarios(n, srb):
        p = tmp_path / (name + ".bin")
        p.write_bytes(encode(batch))
        calls.append({"path": str(p), "srb": srb.hex(), "chunks": chunks, "scalars": r if explicit else None})
        wants.append(reference(batch, r))
    jobs = tmp_path / "jobs.json"
    jobs.write_text(json.dumps({"n": n, "calls": calls}))
    r = subprocess.run([sys.executable, "-c", _CHILD, ROOT, str(jobs)], env=dict(os.environ, **env), capture_output=True,
                       text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    got = [(ok, bytes.fromhex(g)) for ok, g in json.loads(r.stdout.strip().splitlines()[-1])]
    for (name, *_), g, w in zip(scenarios(n, srb), got, wants):
        assert g == w, name


def _to_device(raw):
    import torch
    d = torch.frombuffer(bytearray(raw), dtype=torch.uint8).cuda()
    torch.cuda.synchronize()
    return d


def _finalize_dev(cache, partials, flags=None):
    import nim_blscurve_b200 as bg
    d = _to_device(partials)
    df = None
    if flags is not None:
        import torch
        df = torch.tensor(flags, dtype=torch.int32, device="cuda")
        torch.cuda.synchronize()
    gt = (C.c_uint8 * 576)()
    rc = bg.lib().blsgpu_finalize_dev(cache.handle, C.c_void_p(d.data_ptr()), len(partials) // 576,
                                      C.c_void_p(df.data_ptr()) if df is not None else None, gt)
    return rc, bytes(gt)


@gpu
@pytest.mark.parametrize("world", [3, 8])
def test_degenerate_shares(cache, br, srb, world):
    """Rank shares of one batch: one whose signature sum cancels, one whose signatures are all infinite, and (second
    batch) one with an infinite key, whose partial is sealed.  blsgpu_finalize and blsgpu_finalize_dev over the partials
    give the one-context verdict and GT, and each unsealed partial has the final exponentiation of br.partial."""
    import nim_blscurve_b200 as bg
    be = bg.GpuBackend(cache)
    n = 5 * world
    r = pr.rlc_scalars(srb, n, 0)
    shares = [bg.shard_range(n, world, k) for k in range(world)]
    batch = valid(n)
    f0, c0 = shares[0]
    cs = [TABLE[i % len(TABLE)] for i in range(c0 - 1)]
    cs.append(solve_last(r[f0:f0 + c0], cs))
    for i, cc in zip(range(f0, f0 + c0), cs):
        batch[i] = batch[i][:2] + (("X", cc),)
    f1, c1 = shares[1]
    for i in range(f1, f1 + c1):
        batch[i] = batch[i][:2] + (None,)
    keyed = list(batch)
    keyed[shares[2][0] + 1] = (None,) + keyed[shares[2][0] + 1][1:]
    for b, sealed in ((batch, False), (keyed, True)):
        raw = encode(b)
        want = reference(b, r)
        assert want[0] is False
        assert cache.verify_raw(raw, srb, 0, want_gt=True) == want
        parts, flags = [], []
        for first, cnt in shares:
            p, f = be.partial(raw[first * 320:(first + cnt) * 320], first, n, srb, 0)
            parts.append(p)
            flags.append(f)
        assert flags == [1 if sealed and k == 2 else 0 for k in range(world)]
        if sealed:
            assert parts[2] == ZERO_GT
        else:
            for (first, cnt), p in zip(shares, parts):
                ref_part = br.partial(raw[first * 320:(first + cnt) * 320], first, n, srb, 0)[0]
                assert be.finalize(p) == br.finalize(ref_part), first
        assert be.finalize(b"".join(parts)) == want
        rc, gt = _finalize_dev(cache, b"".join(parts))
        assert (rc, gt) == (int(want[0]), want[1])
        rc, gt = _finalize_dev(cache, b"".join(parts), flags)
        assert (rc, gt) == (int(want[0]), want[1])


def _f12_mem(a):
    return b"".join(pr.fp_to_mont_bytes(x) for j in range(2) for i in range(3) for x in a[j][i])


def _rand_f2(rng):
    return (rng.randrange(pr.P), rng.randrange(pr.P))


def partial_sets(count, rng):
    """kind -> count Fp12 partials"""
    def f12():
        return (tuple(_rand_f2(rng) for _ in range(3)), tuple(_rand_f2(rng) for _ in range(3)))
    zero = (pr.F6_ZERO, pr.F6_ZERO)
    rand = [f12() for _ in range(count)]
    fs = [f12() for _ in range(count // 2)]
    return {"random": rand,
            "one": [pr.F12_ONE] * count,
            "zero_in_one_slot": rand[:count // 2] + [zero] + rand[count // 2 + 1:],
            "fp6": [(f12()[0], pr.F6_ZERO) for _ in range(count)],
            "f_and_conj": [x for f in fs for x in (f, pr.f12_conj(f))] + [pr.F12_ONE] * (count % 2)}


def expected_final(parts):
    acc = pr.F12_ONE
    for x in parts:
        acc = pr.f12_mul(acc, x)
    if acc == (pr.F6_ZERO, pr.F6_ZERO):
        return False, ZERO_GT                    # zero has no inverse: the library maps it to zero, not one
    out = pr.final_exp(acc)
    return out == pr.F12_ONE, pr.f12_to_bytes(out)


@gpu
@pytest.mark.parametrize("count", [1, 2, 3, 7, 8, 9, 63, 64])
def test_finalize_arbitrary_partials(cache, count):
    """blsgpu_finalize on arbitrary Fp12 partials == pyref.final_exp of their product: random elements, ones, a zero
    partial, elements of Fp6 and pairs f, conj(f) (both mapped to one); 65 partials are an argument error"""
    import nim_blscurve_b200 as bg
    be = bg.GpuBackend(cache)
    for kind, parts in partial_sets(count, random.Random(count)).items():
        want = expected_final(parts)
        if kind in ("one", "fp6", "f_and_conj"):
            assert want == (True, ONE_GT)
        assert be.finalize(b"".join(_f12_mem(x) for x in parts)) == want, kind
    gt = (C.c_uint8 * 576)()
    assert bg.lib().blsgpu_finalize(cache.handle, bytes(65 * 576), 65, gt) == ERR_ARG


@gpu
@pytest.mark.parametrize("count", [9, 25, 65, 256])
def test_finalize_dev_many_partials(cache, count):
    """blsgpu_finalize_dev has no upper limit on the partials: past the counts the final-exponentiation programs take
    directly, the partials are folded first, with the same result; a flagged share still rejects the batch"""
    rng = random.Random(1000 + count)
    for kind, parts in partial_sets(count, rng).items():
        want = expected_final(parts)
        raw = b"".join(_f12_mem(x) for x in parts)
        assert _finalize_dev(cache, raw) == (int(want[0]), want[1]), kind
    flags = [0] * count
    flags[count - 1] = 1
    assert _finalize_dev(cache, b"".join(_f12_mem(pr.F12_ONE) for _ in range(count)), flags) == (0, ZERO_GT)
