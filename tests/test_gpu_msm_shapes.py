"""The G1 and G2 Pippenger MSM (msm.cuh) at every window shape route.hpp picks, against references with known discrete
logarithms.

If P_i = [d_i]G, then sum_i [s_i]P_i = [sum_i d_i (s_i mod 2^nbits) mod r]G, so one pyref scalar multiplication gives
the expected affine point whatever the number of points.  The points are
* the benchmark's device inputs (blsgpu_msm_make_inputs: P_i = [k_i]G1 with the 96-bit k_i of a splitmix recipe, which
  is restated here in numpy) for the G1 sizes up to 2^22;
* a progression Q_j = [a + j b]G built in pyref by affine additions for host inputs and for every G2 input; -Q_j has
  the discrete log -(a + j b), the all-zero point is infinity, and larger inputs tile the progression.

The sizes are the first and the last n of every run of equal MSM shape (hostsim hs_msm_runs over route::plan_msm), so a
moved threshold moves them.  After every MSM on a single-device context, the launch count shows whether the window
Horner ran as a dataflow program or as k_msm_horner.  The BLSGPU_MSM_* overrides are read once per process, so the
non-default shapes run in child processes.  A CPU test pins the reference to pyref's sum of scalar multiplications."""
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
from oracle import replay

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
Q = pr.R_ORDER
ERR_ARG = -2                                     # include/blsgpu.h
NBITS = (1, 8, 9, 63, 64, 65, 128, 200, 254, 255, 256)
G1_MAX = 1 << 22                                 # BASELINE configs: the companion G1 MSM up to 2^22 points
B200_SMS = 148
POOL = 1 << 15                                   # points of each progression
SEED = 0x5EED
gpu = pytest.mark.gpu


def g2_max(nbits):
    """64-bit G2 MSMs are the batch's signature sum (up to the context size: 2^18 covers the 131 072 sets per GPU of
    the benchmark); 255 bits is the widest common use; the other widths are covered up to 2^12 points."""
    return 1 << 18 if nbits in (64, 255) else 1 << 12


# ---- shapes from route.hpp -----------------------------------------------------------------------------------------
@functools.lru_cache(maxsize=None)
def _hostsim():
    so = os.path.join(HERE, "hostsim", "libhostsim.so")
    src = os.path.join(HERE, "hostsim", "hostsim.cpp")
    csrc = os.path.join(ROOT, "nim_blscurve_b200", "csrc")
    deps = [src] + [os.path.join(csrc, f) for f in os.listdir(csrc) if f.endswith((".cuh", ".hpp"))]
    if not os.path.exists(so) or any(os.path.getmtime(d) > os.path.getmtime(so) for d in deps):
        subprocess.run(["g++", "-O2", "-shared", "-fPIC", "-x", "c++", "-std=c++17", "-o", so, src], check=True)
    return C.CDLL(so)


def plan(n, nbits, sms):
    """route::plan_msm under the thresholds of the current environment (hostsim.cpp hs_plan_msm)"""
    o = (C.c_longlong * 37)()
    _hostsim().hs_plan_msm(C.c_size_t(n), nbits, sms, o)
    p = dict(zip(("c", "nwin", "B", "L", "nseg", "G", "emax", "horner_prog"), o[:8]))
    p["K"] = list(o[11 + p["G"]:11 + 2 * p["G"]])
    return p


def shape(p):
    return (p["c"], p["nwin"], p["L"], p["nseg"], p["G"], p["horner_prog"], tuple(k == 8 for k in p["K"]))


@functools.lru_cache(maxsize=None)
def msm_runs(nbits, sms, n_max):
    """[(first n, last n)] of every run of equal shape over 1 .. n_max points"""
    cap = 4096
    o = (C.c_longlong * (2 * cap))()
    k = _hostsim().hs_msm_runs(nbits, sms, C.c_size_t(n_max), o, cap)
    assert 0 < k <= cap, k
    return [(o[2 * i], o[2 * i + 1]) for i in range(k)]


def sizes(nbits, sms, n_max):
    return sorted({n for run in msm_runs(nbits, sms, n_max) for n in run})


def expected_launches(p):
    """msm.cuh msm_run: count, three scans and the scatter; per group the chunks, both combines, the segments and the
    levels of the segment tree; then the Horner program (prep, program, finish) or one k_msm_horner per group"""
    levels, m = 0, p["nseg"]
    while m > 1:
        m = (m + 1) // 2
        levels += 1
    return 5 + p["G"] * (4 + levels) + (3 if p["horner_prog"] else p["G"])


# ---- points with known discrete logs -------------------------------------------------------------------------------
# progression of group g2: Q_j = [A + j B]G
PROG = {False: (0x1F0E9D8C7B6A5948372615F4E3D2C1B0A9, 0x6A09E667F3BCC908B2),
        True: (0x3C6EF372FE94F82BA54FF53A5F1D36F1, 0x510E527FADE682D19B)}


def dlog(g2, j, neg=False):
    a, b = PROG[g2]
    return (-(a + j * b) if neg else a + j * b) % Q


_POOLS = {False: [], True: []}


def pool(g2, m):
    """memory bytes of Q_0 .. Q_{m-1}, extended by affine additions as needed"""
    pts = _POOLS[g2]
    if len(pts) < m:
        gen, mul, add, to = (pr.G2_GEN, pr.g2_mul, pr.g2_add, pr.g2_to_mem) if g2 else \
            (pr.G1_GEN, pr.g1_mul, pr.g1_add, pr.g1_to_mem)
        q, step = mul(gen, dlog(g2, len(pts))), mul(gen, PROG[g2][1])
        while len(pts) < m:
            pts.append(to(q))
            q = add(q, step)
    return pts[:m]


def neg_mem(b):
    """-P of an affine point in memory (Montgomery limbs): y -> p - y, coordinate by coordinate"""
    half = len(b) // 2
    ys = [int.from_bytes(b[k:k + 48], "little") for k in range(half, len(b), 48)]
    return b[:half] + b"".join(((pr.P - y) % pr.P).to_bytes(48, "little") for y in ys)


def tiled(g2, n):
    """point i = Q_{i mod POOL}"""
    m = min(n, POOL)
    pts = pool(g2, m)
    return b"".join(pts[i % m] for i in range(n))


# ---- sums of products of large integers as 16-bit limb dot products ------------------------------------------------
def scalar_limbs(raw, n, nbits):
    """n x ceil(sb / 2) 16-bit limbs of the n little-endian scalars of sb = ceil(nbits / 8) bytes in raw, masked to
    nbits bits"""
    sb = (nbits + 7) // 8
    a = np.zeros((n, sb + sb % 2), dtype=np.uint8)
    a[:, :sb] = np.frombuffer(raw, dtype=np.uint8, count=n * sb).reshape(n, sb)
    q, rb = divmod(nbits, 8)
    if q < sb:
        a[:, q] &= (1 << rb) - 1
    return a.view("<u2")


def limb_dot(A, S, lo, hi):
    """[sum_{lo <= i < hi} A_i,c * s_i for every column c of A]: A holds 16-bit coefficients, S the 16-bit limbs of the
    s_i.  Products are below 2^32 and chunks of 2^18 rows keep every sum below 2^53, so float64 products are exact."""
    M = np.zeros((A.shape[1], S.shape[1]), dtype=object)
    for a in range(lo, hi, 1 << 18):
        b = min(hi, a + (1 << 18))
        M += (A[a:b].astype(np.float64).T @ S[a:b].astype(np.float64)).astype(np.int64).astype(object)
    return [sum(int(M[c, j]) << (16 * j) for j in range(S.shape[1])) for c in range(A.shape[1])]


def make_inputs_dlogs(seed, n):
    """the k_i of blsgpu_msm_make_inputs (msm.cuh k_msm_make_inputs): n x 6 16-bit limbs"""
    i = np.arange(n, dtype=np.uint64)
    s = np.uint64(seed) ^ (np.uint64(0xFACADE) + i * np.uint64(0x100000001b3))
    v = []
    for _ in range(2):
        s = s + np.uint64(0x9e3779b97f4a7c15)
        z = (s ^ (s >> np.uint64(30))) * np.uint64(0xbf58476d1ce4e5b9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94d049bb133111eb)
        v.append(z ^ (z >> np.uint64(31)))
    lo = v[0].astype("<u8").view("<u2").reshape(n, 4)
    hi = v[1].astype("<u8").view("<u2").reshape(n, 4)[:, :2]
    return np.ascontiguousarray(np.concatenate([lo, hi], axis=1))


def k_of(K, i):
    return sum(int(K[i, l]) << (16 * l) for l in range(6))


def g1_dlog_sum(K, S, lo, hi):
    return sum(c << (16 * l) for l, c in enumerate(limb_dot(K, S, lo, hi)))


def tiled_dlog_sum(g2, S, lo, hi):
    """sum_i dlog(Q_{i mod POOL}) s_i over [lo, hi)"""
    a, b = PROG[g2]
    A = np.stack([np.ones(hi, dtype=np.uint16), (np.arange(hi) % POOL).astype(np.uint16)], axis=1)
    s0, s1 = limb_dot(A, S, lo, hi)
    return a * s0 + b * s1


def expected(g2, d):
    return pr.g2_to_mem(pr.g2_mul(pr.G2_GEN, d % Q)) if g2 else pr.g1_to_mem(pr.g1_mul(pr.G1_GEN, d % Q))


# ---- scenarios -----------------------------------------------------------------------------------------------------
# A scenario is (name, points, scalars): point i is (j, neg) for +-Q_j or None for infinity; scalar i is an integer
# stored in sb = ceil(nbits / 8) little-endian bytes (taken mod 2^(8 sb)), of which the MSM uses the low nbits bits.
def scenarios(n, nbits, c, m=POOL, seed=0):
    """c: the window width of the plan of (n, nbits)"""
    rng = random.Random(f"{n} {nbits} {c} {seed}")
    sb = (nbits + 7) // 8
    rnd = lambda: rng.getrandbits(nbits)                                   # noqa: E731
    pts = lambda: [(rng.randrange(m), False) for _ in range(n)]            # noqa: E731
    out = [("random", pts(), [rnd() for _ in range(n)]),
           ("zero_scalars", pts(), [0] * n),
           ("points_at_infinity", [None] * n, [rnd() for _ in range(n)])]
    ends = pts()
    ends[0] = ends[-1] = None
    out.append(("infinity_first_and_last", ends, [rnd() for _ in range(n)]))
    pm, sc, rs, sc2 = [], [], [], []                 # (P, -P) with equal scalars; (P, P) with s and r - s
    for i in range(n):
        if i % 2 == 0:
            pm.append((rng.randrange(m), False))
            sc.append(rnd())
            rs.append((rng.randrange(m), False))
            sc2.append(rng.randrange(1, Q))
        else:
            pm.append((pm[-1][0], True))
            sc.append(sc[-1])
            rs.append(rs[-1])
            sc2.append(Q - sc2[-1])
    out += [("plus_minus_equal_scalars", pm, sc), ("s_and_r_minus_s", rs, sc2)]
    one = (rng.randrange(m), False)
    out += [("one_point_random_scalars", [one] * n, [rnd() for _ in range(n)]),
            ("one_point_equal_scalars", [one] * n, [rnd() | 1] * n)]
    special = [0, 1, Q - 1, Q, Q + 1, 1 << (nbits - 1), (1 << nbits) - 1]
    out.append(("special_scalars", pts(), [special[i % len(special)] for i in range(n)]))
    # every raw window value 2^(c-1) or 2^(c-1) + 1: the sign boundary of msm_digit, with and without a carry in
    half = 1 << (c - 1)
    bnd = [sum((half + rng.getrandbits(1)) << (w * c) for w in range(nbits // c + 1)) & ((1 << nbits) - 1)
           for _ in range(n)]
    out.append(("window_sign_boundary", pts(), bnd))
    if 8 * sb > nbits:
        above = ((1 << (8 * sb)) - 1) ^ ((1 << nbits) - 1)
        out.append(("bits_above_nbits", pts(), [rnd() | above for _ in range(n)]))
    return out


def encode(g2, points, scalars, nbits):
    sb = (nbits + 7) // 8
    size = 192 if g2 else 96
    used = {p for p in points if p is not None}
    base = pool(g2, max((j for j, _ in used), default=0) + 1)
    mem = {(j, neg): (neg_mem(base[j]) if neg else base[j]) for j, neg in used}
    pb = b"".join(bytes(size) if p is None else mem[p] for p in points)
    return pb, b"".join((s % (1 << (8 * sb))).to_bytes(sb, "little") for s in scalars)


def reference(g2, points, scalars, nbits):
    """affine memory bytes of sum_i [s_i mod 2^nbits] P_i, by discrete logs"""
    mask = (1 << nbits) - 1
    return expected(g2, sum(dlog(g2, p[0], p[1]) * (s & mask) for p, s in zip(points, scalars) if p is not None))


# ---- CPU -----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("g2", [False, True], ids=["g1", "g2"])
def test_reference_against_pyref_sum(g2):
    """For n <= 8 and every scenario, the discrete-log reference equals pyref's sum of n scalar multiplications
    (oracle/replay.py _ref_msm); so do the limb dot products of the size sweeps, on tiled progressions and on the
    k_i of the make_inputs recipe (restated in numpy, checked against replay.py's splitmix)."""
    for n, nbits in ((1, 255), (2, 9), (7, 64), (8, 256), (8, 1), (7, 63)):
        c = plan(n, nbits, B200_SMS)["c"]
        for name, points, scalars in scenarios(n, nbits, c, m=16):
            pb, sb = encode(g2, points, scalars, nbits)
            assert reference(g2, points, scalars, nbits) == replay._ref_msm(pb, sb, nbits, g2), (n, nbits, name)
    # tiled progression with host scalars, and the G1 make_inputs points
    n, nbits = 8, 65
    sc = bytes(random.Random(3).getrandbits(8) for _ in range(n * 9))
    S = scalar_limbs(sc, n, nbits)
    pts = b"".join(pool(g2, 8)[i % 8] for i in range(n))
    assert expected(g2, tiled_dlog_sum(g2, S, 0, n)) == replay._ref_msm(pts, sc, nbits, g2)
    K = make_inputs_dlogs(SEED, 64)
    for i in range(64):
        s = SEED ^ ((0xFACADE + i * 0x100000001b3) & 0xFFFFFFFFFFFFFFFF)
        s, a = replay._splitmix(s)
        s, b = replay._splitmix(s)
        assert k_of(K, i) == a | (b & 0xFFFFFFFF) << 64, i
    if not g2:
        pts = b"".join(pr.g1_to_mem(pr.g1_mul(pr.G1_GEN, k_of(K, i))) for i in range(n))
        assert expected(False, g1_dlog_sum(K, S, 0, n)) == replay._ref_msm(pts, sc, nbits, False)


def test_combine_scalars_chain():
    """pyref.combine_scalars is the SHA-256 chain of MultiSignatureSet.combine: four little-endian words per digest,
    last word first"""
    srb = hashlib.sha256(b"combine").digest()
    d1 = hashlib.sha256(srb).digest()
    d2 = hashlib.sha256(d1).digest()
    words = [int.from_bytes(d[8 * k:8 * k + 8], "little") for d in (d1, d2) for k in (3, 2, 1, 0)]
    assert pr.combine_scalars(srb, 6) == words[:6]


def test_sizes_reach_every_window_width():
    """The sizes the GPU tests run (first and last n of every run of equal shape) reach every window width the
    default rule picks for each tested nbits, and the nbits = 256 run whose 129 windows keep the Horner off the
    program.  Each run is one shape from its first n to its last, and the next n starts a different one."""
    widths = {}
    for g2, limit in ((False, lambda nb: G1_MAX), (True, g2_max)):
        for nbits in NBITS:
            n_max = limit(nbits)
            runs = msm_runs(nbits, B200_SMS, n_max)
            assert runs[0][0] == 1 and runs[-1][1] == n_max
            assert all(b[0] == a[1] + 1 for a, b in zip(runs, runs[1:]))
            for first, last in runs:
                assert shape(plan(first, nbits, B200_SMS)) == shape(plan(last, nbits, B200_SMS)), (nbits, first, last)
                if last < n_max:
                    assert shape(plan(last + 1, nbits, B200_SMS)) != shape(plan(last, nbits, B200_SMS)), (nbits, last)
            every = {plan(a, nbits, B200_SMS)["c"] for a, _ in runs}
            at = {plan(n, nbits, B200_SMS)["c"] for n in sizes(nbits, B200_SMS, n_max)}
            assert every == at, (g2, nbits)
            widths[("g2" if g2 else "g1", nbits)] = sorted(at)
    # the kernel Horner's default cases: nbits = 256 below 128 points (c = 2, 129 windows)
    kernel = [n for n in sizes(256, B200_SMS, G1_MAX) if not plan(n, 256, B200_SMS)["horner_prog"]]
    assert kernel and all(plan(n, 256, B200_SMS)["nwin"] > 128 for n in kernel), kernel
    for key, w in sorted(widths.items()):
        print(f"{key[0]} nbits={key[1]}: c in {w}")


# ---- GPU -----------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def ctx():
    import nim_blscurve_b200 as bg
    c = bg.BatchedBLSVerifierCache(max_sets=64, device=0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def _dev(raw):
    import torch
    t = torch.frombuffer(bytearray(raw), dtype=torch.uint8).cuda()
    torch.cuda.synchronize()                     # the library's stream does not wait for torch's
    return t


def _fn(g2, dev):
    import nim_blscurve_b200 as bg
    L = bg.lib()
    if g2:
        return L.blsgpu_msm_g2_dev if dev else L.blsgpu_msm_g2
    return L.blsgpu_msm_g1_dev if dev else L.blsgpu_msm_g1


def msm(ctx, sms, g2, points, scalars, n, nbits):
    """one MSM from host buffers (bytes) or device tensors; checks that the window Horner ran as the plan says"""
    import nim_blscurve_b200 as bg
    dev = not isinstance(points, bytes)
    out = (C.c_uint8 * (192 if g2 else 96))()
    args = (C.c_void_p(points.data_ptr()), C.c_void_p(scalars.data_ptr())) if dev else (points, scalars)
    rc = _fn(g2, dev)(ctx.handle, *args, n, nbits, out)
    assert rc == 1, ctx.last_error()
    p = plan(n, nbits, sms)
    assert bg.lib().blsgpu_last_launches(ctx.handle) == expected_launches(p), (n, nbits, p)
    return bytes(out)


@pytest.fixture(scope="module")
def g1_inputs(ctx):
    import torch
    import nim_blscurve_b200 as bg
    dp = torch.empty(G1_MAX * 96, dtype=torch.uint8, device="cuda")
    ds = torch.empty(G1_MAX * 32, dtype=torch.uint8, device="cuda")
    assert bg.lib().blsgpu_msm_make_inputs(ctx.handle, SEED, G1_MAX, C.c_void_p(dp.data_ptr()),
                                           C.c_void_p(ds.data_ptr())) == 0
    return dp, ds, make_inputs_dlogs(SEED, G1_MAX)


@gpu
def test_make_inputs_points(g1_inputs):
    """the benchmark's points are [k_i]G1 for the k_i restated here: the first 64 and a random sample"""
    import torch
    dp, _, K = g1_inputs
    idx = list(range(64)) + sorted(random.Random(7).sample(range(64, G1_MAX), 64))
    rows = dp.view(-1, 96)[torch.tensor(idx, device="cuda")].cpu().numpy()
    for row, i in zip(rows, idx):
        assert row.tobytes() == pr.g1_to_mem(pr.g1_mul(pr.G1_GEN, k_of(K, i))), i


@gpu
@pytest.mark.parametrize("nbits", NBITS)
def test_g1_every_shape(ctx, sms, g1_inputs, nbits):
    """G1, device entry point: the first and the last n of every run of equal shape up to 2^22 points, on prefixes of
    the make_inputs points; 255-bit scalars from make_inputs, other widths seeded host scalars"""
    dp, ds, K = g1_inputs
    ns = sizes(nbits, sms, G1_MAX)
    if nbits == 255:
        raw = ds[:ns[-1] * 32].cpu().numpy().tobytes()
    else:
        raw = np.random.default_rng(nbits).integers(0, 256, ns[-1] * ((nbits + 7) // 8), dtype=np.uint8).tobytes()
        ds = _dev(raw)
    S = scalar_limbs(raw, ns[-1], nbits)
    d, prev, bad = 0, 0, []
    for n in ns:
        d += g1_dlog_sum(K, S, prev, n)
        prev = n
        if msm(ctx, sms, False, dp, ds, n, nbits) != expected(False, d):
            bad.append(n)
    assert not bad, (bad, ns)


@gpu
@pytest.mark.parametrize("nbits", NBITS)
def test_g2_every_shape(ctx, sms, nbits):
    """G2, device entry point: the first and the last n of every run of equal shape up to g2_max(nbits) points of the
    tiled progression, seeded host scalars"""
    ns = sizes(nbits, sms, g2_max(nbits))
    raw = np.random.default_rng(1000 + nbits).integers(0, 256, ns[-1] * ((nbits + 7) // 8), dtype=np.uint8).tobytes()
    dp, ds = _dev(tiled(True, ns[-1])), _dev(raw)
    S = scalar_limbs(raw, ns[-1], nbits)
    d, prev, bad = 0, 0, []
    for n in ns:
        d += tiled_dlog_sum(True, S, prev, n)
        prev = n
        if msm(ctx, sms, True, dp, ds, n, nbits) != expected(True, d):
            bad.append(n)
    assert not bad, (bad, ns)


SMALL_N, LARGE_N = 67, 3001                      # LARGE_N: one bucket of equal scalars holds > MSM_BIG partials


def _run_scenarios(ctx, sms, g2, n, nbits, names=None):
    c = plan(n, nbits, sms)["c"]
    bad = []
    for name, points, scalars in scenarios(n, nbits, c):
        if names and name not in names:
            continue
        pb, sb = encode(g2, points, scalars, nbits)
        want = reference(g2, points, scalars, nbits)
        host = msm(ctx, sms, g2, pb, sb, n, nbits)
        dev = msm(ctx, sms, g2, _dev(pb), _dev(sb), n, nbits)
        if host != want or dev != want:
            bad.append(name)
    assert not bad, bad


@gpu
@pytest.mark.parametrize("n", [SMALL_N, LARGE_N])
@pytest.mark.parametrize("nbits", [64, 255, 256])
@pytest.mark.parametrize("g2", [False, True], ids=["g1", "g2"])
def test_edge_scenarios(ctx, sms, g2, nbits, n):
    """every scenario through the host and the device entry point of its group, byte for byte"""
    _run_scenarios(ctx, sms, g2, n, nbits)


@gpu
@pytest.mark.parametrize("n", [SMALL_N, LARGE_N])
@pytest.mark.parametrize("nbits", [9, 63, 65, 254])
@pytest.mark.parametrize("g2", [False, True], ids=["g1", "g2"])
def test_bits_above_nbits_are_ignored(ctx, sms, g2, nbits, n):
    """bits set above nbits in the last scalar byte (nbits = 255 is among the edge scenarios)"""
    _run_scenarios(ctx, sms, g2, n, nbits, {"bits_above_nbits", "special_scalars", "window_sign_boundary"})


@gpu
@pytest.mark.parametrize("g2", [False, True], ids=["g1", "g2"])
def test_one_bit_scalars(ctx, sms, g2):
    _run_scenarios(ctx, sms, g2, 1 << 16, 1, {"random", "bits_above_nbits", "one_point_random_scalars"})


@gpu
def test_argument_errors(ctx):
    """nbits 0 and 257 are argument errors, n = 0 is an empty sum; the output is zeroed in every case"""
    for g2 in (False, True):
        size = 192 if g2 else 96
        pts, sc = tiled(g2, 3), bytes(range(1, 97))
        dp, ds = _dev(pts), _dev(sc)
        for dev in (False, True):
            args = (C.c_void_p(dp.data_ptr()), C.c_void_p(ds.data_ptr())) if dev else (pts, sc)
            for n, nbits, rc in ((3, 0, ERR_ARG), (3, 257, ERR_ARG), (0, 255, 0)):
                out = (C.c_uint8 * size)(*([0xAB] * size))
                assert _fn(g2, dev)(ctx.handle, *args, n, nbits, out) == rc, (g2, dev, n, nbits)
                assert bytes(out) == bytes(size)


@gpu
def test_multi_device_context_on_one_gpu():
    """blsgpu_create_multi([0, 0, 0]): three shares summed by the leader, one of them cancelling to infinity; below
    2 (1 + peers) = 6 points the leader runs the MSM alone"""
    import nim_blscurve_b200 as bg
    c = bg.BatchedBLSVerifierCache(max_sets=64, devices=[0, 0, 0])
    try:
        for g2 in (False, True):
            for n in (5, 6, 301, 3001):
                rng = random.Random(n)
                points = [(rng.randrange(POOL), False) for _ in range(n)]
                scalars = [rng.getrandbits(255) for _ in range(n)]
                if n >= 6:
                    lo = n // 3 + (1 if n % 3 > 0 else 0)             # share 1 of blsgpu.cu share_range(n, 3, 1)
                    hi = lo + n // 3 + (1 if n % 3 > 1 else 0)
                    for i in range(lo, hi - 1, 2):
                        points[i + 1] = (points[i][0], True)
                        scalars[i + 1] = scalars[i]
                pb, sb = encode(g2, points, scalars, 255)
                got = bg.msmG2(c, pb, sb, 255) if g2 else bg.msmG1(c, pb, sb, 255)
                assert got == reference(g2, points, scalars, 255), (g2, n)
    finally:
        c.close()


@gpu
@pytest.mark.parametrize("n", [1, 2, 5, 4097])
def test_combine(ctx, sms, n):
    """blsgpu_combine: sum [s_i] pk_i and sum [s_i] sig_i with the scalars of the SHA-256 chain; one set is copied"""
    import nim_blscurve_b200 as bg
    srb = hashlib.sha256(b"combine %d" % n).digest()
    js = [(7 * i + 3) % POOL for i in range(n)]
    pks = b"".join(pool(False, POOL)[j] for j in js)
    sigs = b"".join(pool(True, POOL)[j] for j in js)
    pk, sig = (C.c_uint8 * 96)(), (C.c_uint8 * 192)()
    L = bg.lib()
    assert L.blsgpu_combine(ctx.handle, srb, pks, sigs, n, pk, sig) == 1, ctx.last_error()
    if n == 1:
        assert (bytes(pk), bytes(sig)) == (pks, sigs)
        return
    sc = pr.combine_scalars(srb, n)
    assert bytes(pk) == expected(False, sum(dlog(False, j) * s for j, s in zip(js, sc)))
    assert bytes(sig) == expected(True, sum(dlog(True, j) * s for j, s in zip(js, sc)))
    assert L.blsgpu_last_launches(ctx.handle) == 1 + 2 * expected_launches(plan(n, 64, sms))


# ---- the non-default shapes, one child process per configuration ---------------------------------------------------
# the BLSGPU_MSM_* configurations whose plans tests/golden/route_plans.json pins
CHILD_ENVS = [{"BLSGPU_MSM_GROUPS": "4"}, {"BLSGPU_MSM_GROUPS": "9"}, {"BLSGPU_MSM_L": "1"}, {"BLSGPU_MSM_L": "64"},
              {"BLSGPU_MSM_K": "1"}, {"BLSGPU_MSM_C": "8"}, {"BLSGPU_MSM_HORNER_PROG": "0"},
              {"BLSGPU_MSM_C": "13", "BLSGPU_MSM_L": "8", "BLSGPU_MSM_GROUPS": "3", "BLSGPU_MSM_K": "24"}]
CHILD_N = (1, 3, 64, 1000, 5000, 65536)
K1_MAX = {False: 1 << 16, True: 1 << 14}         # K = 1 makes every entry its own partial


@functools.lru_cache(maxsize=None)
def child_cases(k1):
    """[(g2, n, nbits, label, points, scalars, expected)]"""
    cases = []
    for g2 in (False, True):
        top = K1_MAX[g2] if k1 else max(CHILD_N)
        ns = sorted({min(n, top) for n in CHILD_N})
        big = tiled(g2, ns[-1])
        size = 192 if g2 else 96
        for n in ns:
            for nbits in (64, 255):
                rng = random.Random(n * 7 + nbits)
                sc = [rng.getrandbits(nbits) for _ in range(n)]
                pts = [(i % POOL, False) for i in range(n)]
                sb = b"".join(s.to_bytes((nbits + 7) // 8, "little") for s in sc)
                cases.append((g2, n, nbits, "random", big[:n * size], sb, reference(g2, pts, sc, nbits)))
        for n in (64, 5000):
            for nbits in (64, 255):
                for name, pts, sc in scenarios(n, nbits, 8, seed=1):
                    if name in ("plus_minus_equal_scalars", "one_point_random_scalars", "one_point_equal_scalars"):
                        pb, sb = encode(g2, pts, sc, nbits)
                        cases.append((g2, n, nbits, name, pb, sb, reference(g2, pts, sc, nbits)))
    return cases


_CHILD = r'''
import ctypes as C, json, sys
sys.path.insert(0, sys.argv[1])
import nim_blscurve_b200 as bg
L = bg.lib()
c = bg.BatchedBLSVerifierCache(max_sets=64, device=0)
out = []
for j in json.load(open(sys.argv[2])):
    pts, sc = open(j["points"], "rb").read(), open(j["scalars"], "rb").read()
    res = (C.c_uint8 * (192 if j["g2"] else 96))()
    rc = (L.blsgpu_msm_g2 if j["g2"] else L.blsgpu_msm_g1)(c.handle, pts, sc, j["n"], j["nbits"], res)
    out.append([rc, bytes(res).hex(), L.blsgpu_last_launches(c.handle), c.last_error() if rc != 1 else ""])
c.close()
print(json.dumps(out))
'''


@gpu
@pytest.mark.parametrize("env", CHILD_ENVS, ids=lambda e: "_".join(f"{k[11:]}{v}" for k, v in e.items()))
def test_overridden_shapes_in_a_child_process(tmp_path, sms, monkeypatch, env):
    """G1 and G2 from the host entry points under each pinned BLSGPU_MSM_* override: random scalars of 64 and 255
    bits at 1 .. 65 536 points, and the cancelling and repeated-point scenarios; results and launch counts"""
    cases = child_cases(env.get("BLSGPU_MSM_K") == "1")
    jobs = []
    for k, (g2, n, nbits, name, pb, sb, _) in enumerate(cases):
        (tmp_path / f"p{k}").write_bytes(pb)
        (tmp_path / f"s{k}").write_bytes(sb)
        jobs.append({"g2": g2, "n": n, "nbits": nbits, "points": str(tmp_path / f"p{k}"),
                     "scalars": str(tmp_path / f"s{k}")})
    (tmp_path / "jobs.json").write_text(json.dumps(jobs))
    r = subprocess.run([sys.executable, "-c", _CHILD, ROOT, str(tmp_path / "jobs.json")], env=dict(os.environ, **env),
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    got = json.loads(r.stdout.strip().splitlines()[-1])
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    bad = []
    for (g2, n, nbits, name, _, _, want), (rc, out, launches, err) in zip(cases, got):
        case = ("g2" if g2 else "g1", n, nbits, name)
        if rc != 1 or bytes.fromhex(out) != want:
            bad.append(("result",) + case + (rc, err))
        elif launches != expected_launches(plan(n, nbits, sms)):
            bad.append(("launches",) + case + (launches, expected_launches(plan(n, nbits, sms))))
    assert len(got) == len(cases) and not bad, bad
