"""The device field primitives one at a time (blsgpu_test_field) against integer arithmetic, at the inputs that reach
the bounds their comments state: every Montgomery reduction multiplier 0xffffffff, maximal dot-product totals, results
on both sides of the final subtraction, and the quotient step of the device lin_finish at every boundary of its range.

Each input family is plain Python and its claimed property is checked on the CPU here (so are the hostsim build of the
same headers, a model of the device quotient step, and the PTX generator).  The GPU tests compare canonical bytes with
Python integers (Fp) and oracle/pyref.py (Fp2, Fp12), and name the family of every mismatch."""
import ctypes as C
import json
import os
import random
import struct
import subprocess
import sys
import zlib

import pytest

from oracle import pyref as pr

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
P = pr.P
R = 1 << 384
RINV = pow(R, -1, P)
NPINV = (-pow(P, -1, R)) % R          # Montgomery multiplier of a product T: M = T * NPINV mod 2^384
INV2 = pow(2, -1, P)
M32 = 0xffffffff
N_RANDOM = 1 << 16
N_RANDOM_F12 = 1 << 14
N_RANDOM_EXP = 1 << 12               # ops whose Python reference is a full exponentiation
SHAPES = (1, 2, 5, 31, 32, 33, 129, 1000)

# op number, input field elements, input words, output field elements, output words (include/blsgpu.h)
OPS = {
    "fp_mul": (0, 2, 0, 1, 0), "fp_mul_ni": (1, 2, 0, 1, 0), "fp_sqr": (2, 1, 0, 1, 0), "fp_sqr_ni": (3, 1, 0, 1, 0),
    "fp_add": (4, 2, 0, 1, 0), "fp_sub": (5, 2, 0, 1, 0), "fp_neg": (6, 1, 0, 1, 0), "fp_inv": (7, 1, 0, 1, 0),
    "fp_inv_vartime": (8, 1, 0, 1, 0), "fp_pow_p34": (9, 1, 0, 1, 0), "fp_from_mont": (10, 1, 0, 1, 0),
    "fp_parity": (11, 1, 0, 0, 1), "fp_is_lexically_largest_canon": (12, 1, 0, 0, 1),
    "fp2_mul": (13, 4, 0, 2, 0), "fp2_sqr": (14, 2, 0, 2, 0), "fp2_mul_xi": (15, 2, 0, 2, 0), "fp2_mul_fp": (16, 3, 0, 2, 0),
    "fp2_inv": (17, 2, 0, 2, 0), "fp2_inv_vartime": (18, 2, 0, 2, 0), "fp2_rsqrt_or_z": (19, 2, 0, 2, 1),
    "fp2_sgn0": (20, 2, 0, 0, 1), "fp2_is_lexically_largest": (21, 2, 0, 0, 1),
    "h_mul": (22, 4, 0, 2, 0), "h_sqr": (23, 2, 0, 2, 0), "h_mul_xi": (24, 2, 0, 2, 0), "h_mul_fp": (25, 3, 0, 2, 0),
    "h_conj": (26, 2, 0, 2, 0), "h_inv": (27, 2, 0, 2, 0),
    "team_dot3": (28, 6, 0, 1, 0), "team_dot4": (29, 8, 2, 1, 0), "team_mul_line": (30, 18, 0, 12, 0),
    "team_square": (31, 12, 0, 12, 0), "lin_finish": (32, 14, 14, 1, 0),
}
# the masks of team_square's table (acc_team.cuh DBL / ZERO): even coefficients, odd coefficients
SQUARE_MASKS = ((0xc, 0), (0x7, 8))


def mont(x):
    return x * R % P


def canon(raw):
    return raw * RINV % P


def mmul(a, b):
    """Montgomery product of stored values"""
    return a * b * RINV % P


def pre_subtraction(T):
    """t = (T + M p) / 2^384, the value of a Montgomery reduction of T before its final conditional subtraction"""
    return (T + (T * NPINV % R) * P) >> 384


def multiplier(T):
    return T * NPINV % R


# ---- input families (stored Montgomery values, integers < p) -------------------------------------------------------
def edge_values():
    v = [0, 1, 2, P - 1, P - 2, (P - 1) // 2, (P + 1) // 2]
    for j in range(13):                                   # the limb edges below p
        v += [(1 << k) for k in (32 * j - 1, 32 * j, 32 * j + 31) if 0 <= k <= 380]
    v += [P - (1 << (32 * k)) for k in range(12)]
    v += [(R - 1) % P, sum(M32 << (64 * i) for i in range(6)) % P, sum(M32 << (64 * i + 32) for i in range(6)) % P]
    return sorted(set(v))


EDGE = edge_values()


def allones_pairs(rng, count):
    """(a, b), a, b < p, with a b = p (mod 2^384): every reduction multiplier digit is 0xffffffff"""
    out = []
    while len(out) < count:
        a = rng.randrange(1, P, 2)
        b = P * pow(a, -1, R) % R
        if b < P:
            out.append((a, b))
    return out


def _sqrt_mod_2k(x, k=384):
    """the four square roots of an x = 1 (mod 8) modulo 2^k"""
    r = 1
    for i in range(3, k):
        if ((r * r - x) >> i) & 1:
            r += 1 << (i - 1)
    m = 1 << k
    return sorted({r % m, -r % m, (r + (m >> 1)) % m, (-r + (m >> 1)) % m})


def allones_squares(count):
    """a < p with a^2 = u p (mod 2^384) for small u = 3 (mod 8): a^2 = p is impossible (p = 3 mod 8); the multiplier is
    2^384 - u, so every digit but the lowest is 0xffffffff"""
    out = []
    u = 3
    while len(out) < count:
        out += [(a, u) for a in _sqrt_mod_2k(u * P % R) if a < P]
        u += 8
    return out[:count]


def dot_allones(rng, count, k, fixed_rest=True):
    """k-term tuples (a_t, b_t) < p with sum a_t b_t = p (mod 2^384); the other terms at p - 1 or random"""
    out = []
    while len(out) < count:
        rest = [(P - 1, P - 1) if fixed_rest else (rng.randrange(P), rng.randrange(P)) for _ in range(k - 1)]
        a0 = rng.randrange(1, P, 2)
        b0 = (P - sum(x * y for x, y in rest)) * pow(a0, -1, R) % R
        if b0 < P:
            out.append([(a0, b0)] + rest)
    return out


# ---- lin_finish: D = P - N + 128 p, the device quotient step -------------------------------------------------------
LIN_MAXT, LIN_MAXMAG = 7, 15
D_MIN, D_MAX = 128 * P - LIN_MAXT * LIN_MAXMAG * (P - 1), 128 * P + LIN_MAXT * LIN_MAXMAG * (P - 1)


def device_quotient(D):
    """fplin.cuh lin_finish (device form): h = D >> 368, q = umulhi(h, 1321131424) >> 11"""
    h = D >> 368
    return ((h * 1321131424) >> 32) >> 11


def lin_terms(V, rng):
    """positive and negative (x, m) lists, x < p, 1 <= m <= 15, at most 7 each, with sum_pos m x - sum_neg m x = V"""
    if V < 0:
        pos, neg = lin_terms(-V, rng)
        return neg, pos
    X = -(-V // LIN_MAXMAG)
    c = max(1, -(-X // (P - 1)))
    c = rng.randint(c, LIN_MAXT) if X else 0
    pos = []
    for i in range(c):
        x = X // c + (1 if i < X % c else 0)
        pos.append((x, LIN_MAXMAG))
    e = LIN_MAXMAG * X - V
    return pos, ([(e, 1)] if e else [])


def lin_boundary_D():
    """D = kp - 1, kp, kp + 1 for every k the range allows; D on both sides of every h = D >> 368 that is a multiple of
    6658; both extremes"""
    Ds = []
    for k in range(D_MIN // P, D_MAX // P + 2):
        Ds += [k * P + d for d in (-1, 0, 1)]
    for j in range((D_MIN >> 368) // 6658, (D_MAX >> 368) // 6658 + 2):
        Ds += [((j * 6658) << 368) + d for d in (-1, 0, (1 << 368) - 1)]
    Ds += [D_MIN, D_MAX]
    return sorted({D for D in Ds if D_MIN <= D <= D_MAX})


def lin_record(pos, neg):
    xs = [x for x, _ in pos] + [0] * (LIN_MAXT - len(pos)) + [x for x, _ in neg] + [0] * (LIN_MAXT - len(neg))
    ms = [m for _, m in pos] + [0] * (LIN_MAXT - len(pos)) + [m for _, m in neg] + [0] * (LIN_MAXT - len(neg))
    return tuple(xs), tuple(ms)


def lin_value(rec):
    xs, ms = rec
    return sum(x * m for x, m in zip(xs[:7], ms[:7])) - sum(x * m for x, m in zip(xs[7:], ms[7:]))


# ---- families per op: lists of (family name, records); a record is (field elements, words) ------------------------
def _pairs_edge():
    return [((a, b), ()) for a in EDGE for b in EDGE]


def _edge_out_mul(rng):
    recs = []
    for a in EDGE[1:] + [rng.randrange(1, P) for _ in range(64)]:
        for target in (0, 1, P - 1):
            recs.append(((a, target * R * pow(a, -1, P) % P), ()))
    return recs


def families(name, rng):
    F = []
    nr = N_RANDOM_EXP if name in ("fp_pow_p34", "fp2_rsqrt_or_z") else N_RANDOM
    if name in ("fp_mul", "fp_mul_ni"):
        ao = allones_pairs(rng, 1024)
        F += [("edge", _pairs_edge()), ("allones", [((a, b), ()) for a, b in ao] + [((b, a), ()) for a, b in ao]),
              ("max", [((P - 1, P - 1), ())]), ("edge_out", _edge_out_mul(rng))]
    elif name in ("fp_sqr", "fp_sqr_ni"):
        r = pow(2, 192, P)
        F += [("edge", [((a,), ()) for a in EDGE]), ("allones", [((a,), ()) for a, _ in allones_squares(256)]),
              ("edge_out", [((0,), ()), ((r,), ()), ((P - r,), ())])]
    elif name in ("fp_add", "fp_sub"):
        sign = 1 if name == "fp_add" else -1
        F += [("edge", _pairs_edge()),
              ("edge_out", [((a, sign * (t - a) % P), ()) for a in EDGE for t in (0, 1, P - 1)])]
    elif name == "fp2_mul":
        ao = allones_pairs(rng, 768)
        recs = []
        for i in range(0, 768, 3):          # a0 b0, a1 b1 and (a0 + a1)(b0 + b1) with all-ones multipliers
            (a0, b0), (a1, b1), (s0, s1) = ao[i], ao[i + 1], ao[i + 2]
            recs.append(((a0, a1, b0, b1), ()))
            x0, y0 = rng.randrange(P), rng.randrange(P)
            recs.append(((x0, (s0 - x0) % P, y0, (s1 - y0) % P), ()))
        F += [("edge", [((a, b, c, d), ()) for a, b in zip(EDGE, EDGE[::-1]) for c, d in zip(EDGE[3:], EDGE)]),
              ("allones", recs), ("max", [((P - 1,) * 4, ())])]
    elif name in ("fp2_sqr", "h_sqr"):
        # (a0 + a1)(a0 - a1) and a0 a1 with all-ones multipliers
        ao = allones_pairs(rng, 512)
        recs = [(((u + v) * INV2 % P, (u - v) * INV2 % P), ()) for u, v in ao[:256]] + [((a, b), ()) for a, b in ao[256:]]
        F += [("edge", _pairs_edge()), ("allones", recs)]
    elif name == "h_mul":
        # even lane: a0 b0 + (-a1) b1 = p, odd lane: a0 b1 + a1 b0 = p (mod 2^384)
        even, odd = [], []
        while len(even) < 512:
            a0, a1, b1 = rng.randrange(1, P, 2), rng.randrange(P), rng.randrange(P)
            b0 = (P - (P - a1) % P * b1) * pow(a0, -1, R) % R
            if b0 < P:
                even.append(((a0, a1, b0, b1), ()))
        while len(odd) < 512:
            a0, a1, b1 = rng.randrange(P), rng.randrange(1, P, 2), rng.randrange(P)
            b0 = (P - a0 * b1) * pow(a1, -1, R) % R
            if b0 < P:
                odd.append(((a0, a1, b0, b1), ()))
        F += [("edge", [((a, b, c, d), ()) for a, b in zip(EDGE, EDGE[::-1]) for c, d in zip(EDGE[3:], EDGE)]),
              ("allones_even", even), ("allones_odd", odd), ("max", [((P - 1,) * 4, ()), ((P - 1, 1, P - 1, P - 1), ())])]
    elif name in ("fp2_mul_fp", "h_mul_fp"):
        ao = allones_pairs(rng, 256)
        F += [("edge", [((a, b, k), ()) for a, b in zip(EDGE, EDGE[::-1]) for k in EDGE]),
              ("allones", [((a, rng.randrange(P), b), ()) for a, b in ao])]
    elif name.startswith(("fp2_", "h_")):
        F += [("edge", _pairs_edge())]
    elif name == "team_dot3":
        t = dot_allones(rng, 512, 3) + dot_allones(rng, 512, 3, fixed_rest=False)
        F += [("allones", [(tuple(x for x, _ in d) + tuple(y for _, y in d), ()) for d in t]),
              ("max", [((P - 1,) * 6, ())]),
              ("edge", [((a, b, c, d, e, f), ()) for a, b, c in zip(EDGE, EDGE[1:], EDGE[2:])
                        for d, e, f in zip(EDGE[::-1], EDGE[-2::-1], EDGE[-3::-1])])]
    elif name == "team_dot4":
        recs = []
        for dbl, zero in SQUARE_MASKS:
            for d in dot_allones(rng, 256, 4) + dot_allones(rng, 256, 4, fixed_rest=False):
                # register side as stored: halved where the kernel doubles it, anything where it is zeroed
                a = [rng.randrange(P) if (zero >> t) & 1 else (d[t][0] * INV2 % P if (dbl >> t) & 1 else d[t][0])
                     for t in range(4)]
                if zero:                    # the zeroed term drops out: re-solve the first term without it
                    rest = sum(d[t][0] * d[t][1] for t in range(1, 4) if not (zero >> t) & 1)
                    b0 = (P - rest) * pow(d[0][0], -1, R) % R
                    if b0 >= P:
                        continue
                    d[0] = (d[0][0], b0)
                recs.append((tuple(a) + tuple(y for _, y in d), (dbl, zero)))
        F += [("allones", recs)]
        F += [("max", [((P - 1,) * 8, m) for m in SQUARE_MASKS] + [(((P - 1) // 2,) * 4 + (P - 1,) * 4, m)
                                                                     for m in SQUARE_MASKS + ((0xf, 0),)])]
        F += [("edge", [((a, b, c, d) + (e,) * 4, m) for a, b, c, d in zip(EDGE, EDGE[1:], EDGE[2:], EDGE[3:])
                        for e in (P - 1, 1) for m in SQUARE_MASKS])]
        F += [("random", [(tuple(rng.randrange(P) for _ in range(8)), (rng.randrange(16), rng.randrange(16)))
                          for _ in range(N_RANDOM)])]
        return F
    elif name in ("team_mul_line", "team_square"):
        one = tuple(mont(1) if i == 0 else 0 for i in range(12))
        fs = [("f_one", one), ("f_zero", (0,) * 12), ("f_max", (P - 1,) * 12)]
        fs += [("f_edge", tuple(EDGE[(i * 7 + j) % len(EDGE)] for j in range(12))) for i in range(len(EDGE))]
        fs += [("random", tuple(rng.randrange(P) for _ in range(12))) for _ in range(N_RANDOM_F12)]
        by = {}
        for i, (fam, f) in enumerate(fs):
            if name == "team_square":
                by.setdefault(fam, []).append((f, ()))
                continue
            by.setdefault(fam, []).append((f + tuple(rng.randrange(P) for _ in range(6)), ()))
            if fam != "random" or i % 64 == 0:
                by.setdefault(fam + "+line_neutral", []).append((f + (mont(1), 0, 0, 0, 0, 0), ()))
                by.setdefault(fam + "+line_max", []).append((f + (P - 1,) * 6, ()))
        return sorted(by.items())
    elif name == "lin_finish":
        bnd = []
        for D in lin_boundary_D():
            bnd.append(lin_record(*lin_terms(D - 128 * P, rng)))
        ext = [lin_record([(P - 1, 15)] * 7, []), lin_record([], [(P - 1, 15)] * 7), lin_record([], []),
               lin_record([(P - 1, 15)] * 7, [(P - 1, 15)] * 7)]
        rnd = []
        for _ in range(N_RANDOM):
            pos = [(rng.choice(EDGE) if rng.random() < 0.2 else rng.randrange(P), rng.randint(1, 15))
                   for _ in range(rng.randint(0, 7))]
            neg = [(rng.choice(EDGE) if rng.random() < 0.2 else rng.randrange(P), rng.randint(1, 15))
                   for _ in range(rng.randint(0, 7))]
            rnd.append(lin_record(pos, neg))
        return [("boundary", bnd), ("extreme", ext), ("random", rnd)]
    else:                                   # unary Fp ops
        F += [("edge", [((a,), ()) for a in EDGE])]
    k = OPS[name][1]
    return F + [("random", [(tuple(rng.randrange(P) for _ in range(k)), ()) for _ in range(nr)])]


# ---- references ---------------------------------------------------------------------------------------------------
def _c2(x, i=0):
    return (canon(x[i]), canon(x[i + 1]))


def _m2(a):
    return (mont(a[0]), mont(a[1]))


def _minv(x):
    return R * R * pow(x, -1, P) % P if x else 0


def _f2inv(a):
    return (0, 0) if a == (0, 0) else pr.f2_inv(a)


def _f12(x):
    c = [_c2(x, 2 * s) for s in range(6)]
    return ((c[0], c[1], c[2]), (c[3], c[4], c[5]))


def _f12m(f):
    return tuple(mont(v) for j in range(2) for i in range(3) for v in f[j][i])


def reference(name, rec):
    """(output field elements, output words) of one record"""
    x, w = rec
    if name in ("fp_mul", "fp_mul_ni"):
        return (mmul(x[0], x[1]),), ()
    if name in ("fp_sqr", "fp_sqr_ni"):
        return (mmul(x[0], x[0]),), ()
    if name == "fp_add":
        return ((x[0] + x[1]) % P,), ()
    if name == "fp_sub":
        return ((x[0] - x[1]) % P,), ()
    if name == "fp_neg":
        return ((-x[0]) % P,), ()
    if name in ("fp_inv", "fp_inv_vartime"):
        return (_minv(x[0]),), ()
    if name == "fp_pow_p34":
        return (mont(pow(canon(x[0]), (P - 3) // 4, P)),), ()
    if name == "fp_from_mont":
        return (canon(x[0]),), ()
    if name == "fp_parity":
        return (), (canon(x[0]) & 1,)
    if name == "fp_is_lexically_largest_canon":
        return (), (int(x[0] > (P - 1) // 2),)
    if name in ("fp2_mul", "h_mul"):
        return _m2(pr.f2_mul(_c2(x), _c2(x, 2))), ()
    if name in ("fp2_sqr", "h_sqr"):
        return _m2(pr.f2_sqr(_c2(x))), ()
    if name in ("fp2_mul_xi", "h_mul_xi"):
        return _m2(pr.f2_mul_xi(_c2(x))), ()
    if name in ("fp2_mul_fp", "h_mul_fp"):
        return _m2(pr.f2_muli(_c2(x), canon(x[2]))), ()
    if name in ("fp2_inv", "fp2_inv_vartime", "h_inv"):
        return _m2(_f2inv(_c2(x))), ()
    if name == "h_conj":
        return (x[0], (-x[1]) % P), ()
    if name == "fp2_sgn0":
        return (), (pr.f2_sgn0(_c2(x)),)
    if name == "fp2_is_lexically_largest":
        c = _c2(x)
        return (), (int((c[1] if c[1] else c[0]) > (P - 1) // 2),)
    if name == "team_dot3":
        return (sum(x[t] * x[3 + t] for t in range(3)) * RINV % P,), ()
    if name == "team_dot4":
        dbl, zero = w
        return (sum((0 if (zero >> t) & 1 else (2 if (dbl >> t) & 1 else 1)) * x[t] * x[4 + t]
                    for t in range(4)) * RINV % P,), ()
    if name == "team_mul_line":
        return _f12m(pr.f12_mul(_f12(x), pr._line_sparse(_c2(x, 12), _c2(x, 14), _c2(x, 16)))), ()
    if name == "team_square":
        return _f12m(pr.f12_sqr(_f12(x))), ()
    if name == "lin_finish":
        return (lin_value(rec) % P,), ()
    raise KeyError(name)


def pre_subtraction_totals(name, rec):
    """the integer totals T that the op's Montgomery reductions see (before the final subtraction)"""
    x, w = rec
    if name in ("fp_mul", "fp_mul_ni"):
        return [x[0] * x[1]]
    if name in ("fp_sqr", "fp_sqr_ni"):
        return [x[0] * x[0]]
    if name == "team_dot3":
        return [sum(x[t] * x[3 + t] for t in range(3))]
    if name == "team_dot4":
        dbl, zero = w
        return [sum(0 if (zero >> t) & 1 else ((2 * x[t] % P) if (dbl >> t) & 1 else x[t]) * x[4 + t] for t in range(4))]
    if name == "h_mul":
        return [x[0] * x[2] + (P - x[1]) % P * x[3], x[0] * x[3] + x[1] * x[2]]
    raise KeyError(name)


# ---- packing ------------------------------------------------------------------------------------------------------
def rec_bytes(nfe, nw):
    return 48 * nfe + 16 * ((nw + 3) // 4)


def pack(recs, nfe, nw):
    pad = bytes(16 * ((nw + 3) // 4) - 4 * nw)
    out = bytearray()
    for x, w in recs:
        for v in x:
            out += v.to_bytes(48, "little")
        if nw:
            out += struct.pack("<%dI" % nw, *w) + pad
    return bytes(out)


def unpack(raw, n, nfe, nw):
    rb = rec_bytes(nfe, nw)
    res = []
    for i in range(n):
        r = raw[i * rb:(i + 1) * rb]
        res.append((tuple(int.from_bytes(r[48 * j:48 * j + 48], "little") for j in range(nfe)),
                    struct.unpack_from("<%dI" % nw, r, 48 * nfe) if nw else ()))
    return res


def run(cache, name, recs):
    import nim_blscurve_b200 as bg
    op, nin, niw, nout, now = OPS[name]
    n = len(recs)
    out = (C.c_uint8 * max(1, n * rec_bytes(nout, now)))()
    rc = bg.lib().blsgpu_test_field(cache.handle, op, pack(recs, nin, niw), rec_bytes(nin, niw), n, out,
                                    rec_bytes(nout, now))
    assert rc == 0, (name, rc, cache.last_error())
    return unpack(bytes(out), n, nout, now)


# ---- CPU: the families have the properties they claim ---------------------------------------------------------------
def test_families_have_their_properties():
    rng = random.Random(1)
    assert all(0 <= v < P for v in EDGE) and len(EDGE) > 40
    hits = 0
    for _ in range(20000):
        a = rng.randrange(1, P, 2)
        hits += P * pow(a, -1, R) % R < P
    assert 0.09 < hits / 20000 < 0.13                          # the share of b = p / a (mod 2^384) below p
    for a, b in allones_pairs(rng, 200):
        assert a < P and b < P and a * b % R == P
        assert multiplier(a * b) == R - 1 and pre_subtraction(a * b) >= P
    for a, u in allones_squares(64):
        assert a < P and u % 8 == 3 and a * a % R == u * P % R
        m = multiplier(a * a)
        assert m & M32 == (1 << 32) - u and m >> 32 == (1 << 352) - 1
    for k in (3, 4):
        for d in dot_allones(rng, 50, k) + dot_allones(rng, 50, k, fixed_rest=False):
            T = sum(x * y for x, y in d)
            assert all(x < P and y < P for x, y in d) and T % R == P and multiplier(T) == R - 1
    for name in ("fp2_sqr", "fp2_mul", "h_mul", "team_dot4"):
        fams = dict(families(name, random.Random(2)))
        for x, w in fams["allones" if name != "h_mul" else "allones_even"]:
            if name == "fp2_sqr":
                Ts = [(x[0] + x[1]) % P * ((x[0] - x[1]) % P), x[0] * x[1]]
            elif name == "fp2_mul":
                Ts = [x[0] * x[2], x[1] * x[3], (x[0] + x[1]) % P * ((x[2] + x[3]) % P)]
            else:
                Ts = pre_subtraction_totals(name, (x, w))[:1]
            assert any(T % R == P for T in Ts), (name, x)
    # lin_finish: D = kp - 1, kp, kp + 1 for 24 <= k <= 232, and both sides of the multiples of 6658 in h
    Ds = lin_boundary_D()
    assert D_MIN // P == 23 and D_MAX // P == 232
    ks = {D // P for D in Ds if D % P == 0}
    assert ks == set(range(24, 233))
    assert all(D - 1 in Ds and D + 1 in Ds for D in Ds if D % P == 0)
    hs = {D >> 368 for D in Ds}
    mults = [h for h in range((D_MIN >> 368) + 1, (D_MAX >> 368) + 1) if h % 6658 == 0]
    assert len(mults) > 200 and all(h in hs and h - 1 in hs for h in mults)
    fam = dict(families("lin_finish", random.Random(3)))
    for (xs, ms), D in zip(fam["boundary"], Ds):
        assert all(x < P for x in xs) and all(0 <= m <= 15 for m in ms)
        assert lin_value((xs, ms)) + 128 * P == D
    assert {lin_value(r) + 128 * P for r in fam["extreme"]} >= {D_MIN, D_MAX}


def test_families_reach_both_sides_of_the_final_subtraction():
    for name in ("fp_mul", "fp_sqr", "team_dot3", "team_dot4", "h_mul"):
        fams = families(name, random.Random(4))
        ts = [pre_subtraction(T) for _, recs in fams for r in recs for T in pre_subtraction_totals(name, r)]
        assert min(ts) < P <= max(ts), name
        assert max(ts) < 2 * P, name                           # the single subtraction suffices


def test_device_lin_finish_quotient_step_model():
    """fplin.cuh lin_finish (device form) restated on integers over the boundary family: the estimate never overshoots,
    undershoots by at most 2, and leaves D - q p below 4p for reduce_4p12."""
    assert (P >> 368) == 6657 and 1321131424 == (1 << 43) // 6658
    assert D_MIN > 0 and D_MAX < 233 * P
    Ds = lin_boundary_D()
    rng = random.Random(5)
    Ds += [rng.randrange(D_MIN, D_MAX + 1) for _ in range(20000)]
    under = set()
    for D in Ds:
        q = device_quotient(D)
        assert q * P <= D, hex(D)
        assert D // P - q <= 2, hex(D)
        assert D - q * P < 4 * P, hex(D)
        under.add(D // P - q)
    assert under >= {0, 1}


# ---- CPU: the same families through hostsim's portable build ------------------------------------------------------
@pytest.fixture(scope="module")
def hs():
    so = os.path.join(HERE, "hostsim", "libhostsim.so")
    src = os.path.join(HERE, "hostsim", "hostsim.cpp")
    csrc = os.path.join(ROOT, "nim_blscurve_b200", "csrc")
    deps = [src] + [os.path.join(csrc, f) for f in os.listdir(csrc) if f.endswith((".cuh", ".hpp"))]
    if not os.path.exists(so) or any(os.path.getmtime(d) > os.path.getmtime(so) for d in deps):
        subprocess.run(["g++", "-O2", "-shared", "-fPIC", "-x", "c++", "-std=c++17", "-o", so, src], check=True)
    return C.CDLL(so)


def _b(v):
    return (C.c_uint8 * 48).from_buffer_copy(v.to_bytes(48, "little"))


def _hs_call(fn, *args):
    r = (C.c_uint8 * 48)()
    fn(*[_b(a) for a in args], r)
    return int.from_bytes(bytes(r), "little")


def test_hostsim_on_the_families(hs):
    rng = random.Random(6)
    for name, fn in (("fp_mul", hs.hs_fp_mul), ("fp_add", hs.hs_fp_add), ("fp_sub", hs.hs_fp_sub)):
        for fam, recs in families(name, rng):
            for rec in recs[:4096]:
                assert _hs_call(fn, *rec[0]) == reference(name, rec)[0][0], (name, fam, [hex(v) for v in rec[0]])
    for fam, recs in families("fp_sqr", rng):
        for rec in recs[:4096]:
            assert _hs_call(hs.hs_fp_mul, rec[0][0], rec[0][0]) == reference("fp_sqr", rec)[0][0], (fam, hex(rec[0][0]))
    for name, fn in (("fp_inv", hs.hs_fp_inv), ("fp_inv_vartime", hs.hs_fp_inv_vartime)):
        for fam, recs in families(name, rng):
            for rec in recs[:256]:
                assert _hs_call(fn, rec[0][0]) == reference(name, rec)[0][0], (name, fam, hex(rec[0][0]))
    for fam, recs in families("fp2_rsqrt_or_z", rng):
        for rec in recs[:512]:
            sq, r = _hs_rsqrt(hs, rec[0])
            _check_rsqrt(rec[0], sq, r, fam)


def _hs_rsqrt(hs, x):
    r = (C.c_uint8 * 96)()
    sq = hs.hs_fp2_rsqrt((C.c_uint8 * 96).from_buffer_copy(x[0].to_bytes(48, "little") + x[1].to_bytes(48, "little")), r)
    raw = bytes(r)
    return sq, (int.from_bytes(raw[:48], "little"), int.from_bytes(raw[48:], "little"))


def _check_rsqrt(x, sq, r, fam):
    a = _c2(x)
    assert bool(sq) == pr.f2_is_square(a), (fam, x)
    tgt = a if sq else pr.f2_mul(pr.SSWU_Z, a)
    if tgt != (0, 0):
        assert pr.f2_mul(pr.f2_sqr(_c2(r)), tgt) == (1, 0), (fam, x)
    assert r[0] < P and r[1] < P


# ---- CPU: the PTX generator ---------------------------------------------------------------------------------------
def test_ptx_generator_check_and_committed_output():
    """tools/gen_fp_ptx.py interprets its PTX against big integers (check()), and fp_gen.cuh is exactly its output."""
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    try:
        import gen_fp_ptx
    finally:
        sys.path.pop(0)
    gen_fp_ptx.check()
    with open(os.path.join(ROOT, "nim_blscurve_b200", "csrc", "fp_gen.cuh")) as f:
        assert gen_fp_ptx.render() == f.read()


# ---- GPU ----------------------------------------------------------------------------------------------------------
ELEMENTWISE = [k for k in OPS if k != "fp2_rsqrt_or_z"]


@pytest.mark.gpu
@pytest.mark.parametrize("name", ELEMENTWISE)
def test_field_op_vs_integers(cache, name):
    rng = random.Random(zlib.crc32(name.encode()))
    fams = families(name, rng)
    labels = [fam for fam, recs in fams for _ in recs]
    recs = [r for _, rs in fams for r in rs]
    got = run(cache, name, recs)
    count, first = {}, {}
    for fam, rec, g in zip(labels, recs, got):
        if g != reference(name, rec):
            count[fam] = count.get(fam, 0) + 1
            first.setdefault(fam, ([hex(v) for v in rec[0]], rec[1]))
    assert not count, "%s: mismatches by family %s; first input of each: %s" % (name, count, first)
    # the same records at sizes that leave partial warps, pairs, teams and blocks give the same bytes
    for n in SHAPES + ((7, 23, 41) if name in ("team_mul_line", "team_square") else ()):
        assert run(cache, name, recs[:n]) == got[:n], (name, n)


@pytest.mark.gpu
def test_fp2_rsqrt_or_z_vs_pyref_and_hostsim(cache, hs):
    rng = random.Random(7)
    fams = families("fp2_rsqrt_or_z", rng)
    recs = [r for _, rs in fams for r in rs]
    labels = [fam for fam, rs in fams for _ in rs]
    got = run(cache, "fp2_rsqrt_or_z", recs)
    for fam, rec, (r, (sq,)) in zip(labels, recs, got):
        _check_rsqrt(rec[0], sq, r, fam)
    for i in list(range(len(recs) - N_RANDOM_EXP)) + list(range(len(recs) - N_RANDOM_EXP, len(recs), 16)):
        assert _hs_rsqrt(hs, recs[i][0]) == (got[i][1][0], got[i][0]), (labels[i], recs[i])
    for n in SHAPES:
        assert run(cache, "fp2_rsqrt_or_z", recs[:n]) == got[:n]


@pytest.mark.gpu
def test_field_entry_rejects_wrong_sizes_and_ops(cache):
    import nim_blscurve_b200 as bg
    L = bg.lib()
    buf = (C.c_uint8 * 4096)()
    for name, (op, nin, niw, nout, now) in OPS.items():
        rin, rout = rec_bytes(nin, niw), rec_bytes(nout, now)
        assert L.blsgpu_test_field(cache.handle, op, buf, rin + 16, 1, buf, rout) == -2, name
        assert L.blsgpu_test_field(cache.handle, op, buf, rin, 1, buf, rout - 16 if rout > 16 else rout + 16) == -2, name
    assert L.blsgpu_test_field(cache.handle, len(OPS), buf, 96, 1, buf, 48) == -2
    assert L.blsgpu_test_field(cache.handle, -1, buf, 96, 1, buf, 48) == -2


FORMAT_CHILD = r'''
import ctypes as C, hashlib, json, sys
sys.path.insert(0, %r)
import nim_blscurve_b200 as bg
srb = hashlib.sha256(b"format").digest()
c = bg.BatchedBLSVerifierCache(max_sets=4096, device=0)
L = bg.lib()
res = {}
def sets(seed, n):
    out = (C.c_uint8 * (320 * n))()
    assert L.blsgpu_make_sets(c.handle, seed, 0, n, out, 0) == 0
    return bytes(out)
s = sets(91, 300)
h = (C.c_uint8 * (300 * 288))()
assert L.blsgpu_test_small_hash(c.handle, s, 300, None, h) == 0
res["small_hash"] = bytes(h).hex()
for n in (1, 33, 129, 4096):
    s = sets(92 + n, n)
    ok, gt = c.verify_raw(s, srb, 16, want_gt=True)
    bad = bytearray(s); bad[(n // 2) * 320 + 100] ^= 1
    bok, bgt = c.verify_raw(bytes(bad), srb, 16, want_gt=True)
    res["batch%%d" %% n] = [ok, gt.hex(), bok, bgt.hex()]
s = sets(93, 200)
pk = b"".join(s[320 * i:320 * i + 96] for i in range(200))
sig = b"".join(s[320 * i + 128:320 * i + 320] for i in range(64))
sc = b"".join(hashlib.sha256(b"k%%d" %% i).digest()[:31] + b"\x00" for i in range(200))
res["msm_g1"] = [bg.msmG1(c, pk[:96 * n], sc[:32 * n], nb).hex() for n, nb in ((1, 255), (37, 255), (200, 64))]
res["msm_g2"] = [bg.msmG2(c, sig[:192 * n], sc[:32 * n], nb).hex() for n, nb in ((1, 255), (64, 255), (20, 64))]
res["combine"] = [x.hex() for n in (1, 5) for x in bg.combine(c, srb, [pk[96 * i:96 * i + 96] for i in range(n)],
                                                               [sig[192 * i:192 * i + 192] for i in range(n)])]
c.close()
print(json.dumps(res))
'''


@pytest.mark.gpu
def test_program_format_2_matches_format_1():
    """Format 2 of the dataflow programs (k_fp_program2, _stream, _rows; fplin.cuh lin_finish on the device) against
    format 1: the small-route message hash, small batches valid and with one corrupted set, G1 and G2 MSMs whose window
    Horner runs as a program, and combine, each in a child process with BLSGPU_PROG_FORMAT set."""
    outs = {}
    for fmt in ("1", "2"):
        env = dict(os.environ, BLSGPU_PROG_FORMAT=fmt)
        r = subprocess.run([sys.executable, "-c", FORMAT_CHILD % ROOT], env=env, capture_output=True, text=True,
                           timeout=900)
        assert r.returncode == 0, r.stderr[-3000:]
        outs[fmt] = json.loads(r.stdout.strip().splitlines()[-1])
    one, two = outs["1"], outs["2"]
    for n in (1, 33, 129, 4096):
        ok, _, bok, _ = one["batch%d" % n]
        assert ok is True and bok is False, n
    for k in one:
        assert two[k] == one[k], k
