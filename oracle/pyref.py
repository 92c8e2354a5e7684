"""Pure-Python big-integer restatement of the nim-blscurve batch-verification path.

TEST INFRASTRUCTURE ONLY.  Nothing under ``nim_blscurve_b200/`` may import this
module; it exists so that tests can check the CUDA path and so that
``tools/gen_consts.py`` can derive the Montgomery-form constant tables from
their defining expressions.  It is slow (seconds per pairing) and is meant for
small cases; the bulk oracle is BLST itself (``oracle/_ref``).

Pinned against: RFC 9380 vectors shipped with the reference
(vendor/blst/bindings/vectors/hash_to_curve/*.json) and against BLST outputs
(tests/test_oracle.py).

Reference map (file:line under /root/reference):
  * tower                vendor/blst/src/fp12_tower.c:9-13
  * expand_message_xmd   vendor/blst/src/hash_to_field.c:51-114
  * hash_to_field        vendor/blst/src/hash_to_field.c:120-154
  * SSWU / isogeny / cofactor  vendor/blst/src/map_to_g2.c:173-290, :43-171, :327-349
  * Miller loop          vendor/blst/src/pairing.c:220-261
  * final exponentiation vendor/blst/src/pairing.c:371-404  (power 3*(p^12-1)/r)
  * GT serialisation     vendor/blst/src/fp12_tower.c:773-786
  * RLC scalar chain     blscurve/blst/blst_min_pubkey_sig_core.nim:476-505, :545-556
  * chunking             blscurve/parallel_chunks.nim:42-55
  * batch verify         blscurve/bls_batch_verifier.nim:121-160, :296-371
  * finalverify          vendor/blst/src/aggregate.c:460-501
"""
import hashlib

# ----------------------------------------------------------------------------
# parameters (vendor/blst/src/consts.c:9-31)
Z_ABS = 0xd201000000010000
X = -Z_ABS
P = (X - 1) ** 2 * (X ** 4 - X ** 2 + 1) // 3 + X
R_ORDER = X ** 4 - X ** 2 + 1
assert P == 0x1a0111ea397fe69a4b1ba7b6434bacd764774b84f38512bf6730d2a0f6b0f6241eabfffeb153ffffb9feffffffffaaab
assert R_ORDER == 0x73eda753299d7d483339d80809a1d80553bda402fffe5bfeffffffff00000001
MONT_R = 1 << 384
DST_ETH2 = b"BLS_SIG_BLS12381G2_XMD:SHA-256_SSWU_RO_POP_"  # blscurve/bls_sig_min_pubkey.nim:31


def inv(a, m=P):
    return pow(a, -1, m)


# ----------------------------------------------------------------------------
# Fp2 = Fp[u]/(u^2+1): tuples (c0, c1)
def f2(a, b=0):
    return (a % P, b % P)


F2_ZERO = (0, 0)
F2_ONE = (1, 0)


def f2_add(a, b):
    return ((a[0] + b[0]) % P, (a[1] + b[1]) % P)


def f2_sub(a, b):
    return ((a[0] - b[0]) % P, (a[1] - b[1]) % P)


def f2_neg(a):
    return ((-a[0]) % P, (-a[1]) % P)


def f2_mul(a, b):
    return ((a[0] * b[0] - a[1] * b[1]) % P, (a[0] * b[1] + a[1] * b[0]) % P)


def f2_sqr(a):
    return f2_mul(a, a)


def f2_muli(a, k):
    return (a[0] * k % P, a[1] * k % P)


def f2_conj(a):
    return (a[0], (-a[1]) % P)


def f2_inv(a):
    n = inv((a[0] * a[0] + a[1] * a[1]) % P)
    return (a[0] * n % P, (-a[1]) * n % P)


def f2_pow(a, e):
    r = F2_ONE
    while e:
        if e & 1:
            r = f2_mul(r, a)
        a = f2_sqr(a)
        e >>= 1
    return r


def f2_is_square(a):
    n = (a[0] * a[0] + a[1] * a[1]) % P
    return n == 0 or pow(n, (P - 1) // 2, P) == 1


def fp_sqrt(a):
    s = pow(a, (P + 1) // 4, P)
    return s if s * s % P == a % P else None


def f2_sqrt(a):
    """Any square root of a in Fp2 (complex method), or None."""
    if a == F2_ZERO:
        return F2_ZERO
    a0, a1 = a
    if a1 == 0:
        s = fp_sqrt(a0)
        if s is not None:
            return (s, 0)
        s = fp_sqrt((-a0) % P)
        return (0, s)
    n = fp_sqrt((a0 * a0 + a1 * a1) % P)
    if n is None:
        return None
    half = inv(2)
    t = (a0 + n) * half % P
    x0 = fp_sqrt(t)
    if x0 is None:
        t = (a0 - n) * half % P
        x0 = fp_sqrt(t)
    x1 = a1 * inv(2 * x0) % P
    r = (x0, x1)
    assert f2_sqr(r) == a
    return r


def fp_sgn0(a):
    return a & 1


def f2_sgn0(a):
    # RFC 9380 4.1 ; vendor/blst/src/no_asm.h:538-554
    s0, z0 = a[0] & 1, a[0] == 0
    s1 = a[1] & 1
    return s0 | (z0 & s1)


# ----------------------------------------------------------------------------
# Fp6 = Fp2[v]/(v^3 - (u+1)), Fp12 = Fp6[w]/(w^2 - v)
XI = (1, 1)


def f2_mul_xi(a):
    return ((a[0] - a[1]) % P, (a[0] + a[1]) % P)


F6_ZERO = (F2_ZERO, F2_ZERO, F2_ZERO)
F6_ONE = (F2_ONE, F2_ZERO, F2_ZERO)


def f6_add(a, b):
    return tuple(f2_add(x, y) for x, y in zip(a, b))


def f6_sub(a, b):
    return tuple(f2_sub(x, y) for x, y in zip(a, b))


def f6_neg(a):
    return tuple(f2_neg(x) for x in a)


def f6_mul(a, b):
    a0, a1, a2 = a
    b0, b1, b2 = b
    t0, t1, t2 = f2_mul(a0, b0), f2_mul(a1, b1), f2_mul(a2, b2)
    c0 = f2_add(t0, f2_mul_xi(f2_sub(f2_sub(f2_mul(f2_add(a1, a2), f2_add(b1, b2)), t1), t2)))
    c1 = f2_add(f2_sub(f2_sub(f2_mul(f2_add(a0, a1), f2_add(b0, b1)), t0), t1), f2_mul_xi(t2))
    c2 = f2_add(f2_sub(f2_sub(f2_mul(f2_add(a0, a2), f2_add(b0, b2)), t0), t2), t1)
    return (c0, c1, c2)


def f6_mul_v(a):
    return (f2_mul_xi(a[2]), a[0], a[1])


def f6_inv(a):
    a0, a1, a2 = a
    c0 = f2_sub(f2_sqr(a0), f2_mul_xi(f2_mul(a1, a2)))
    c1 = f2_sub(f2_mul_xi(f2_sqr(a2)), f2_mul(a0, a1))
    c2 = f2_sub(f2_sqr(a1), f2_mul(a0, a2))
    t = f2_add(f2_mul(a0, c0), f2_mul_xi(f2_add(f2_mul(a2, c1), f2_mul(a1, c2))))
    t = f2_inv(t)
    return (f2_mul(c0, t), f2_mul(c1, t), f2_mul(c2, t))


F12_ONE = (F6_ONE, F6_ZERO)


def f12_mul(a, b):
    a0, a1 = a
    b0, b1 = b
    t0, t1 = f6_mul(a0, b0), f6_mul(a1, b1)
    c1 = f6_sub(f6_sub(f6_mul(f6_add(a0, a1), f6_add(b0, b1)), t0), t1)
    c0 = f6_add(t0, f6_mul_v(t1))
    return (c0, c1)


def f12_sqr(a):
    return f12_mul(a, a)


def f12_conj(a):
    return (a[0], f6_neg(a[1]))


def f12_inv(a):
    a0, a1 = a
    t = f6_sub(f6_mul(a0, a0), f6_mul_v(f6_mul(a1, a1)))
    t = f6_inv(t)
    return (f6_mul(a0, t), f6_neg(f6_mul(a1, t)))


def f12_pow(a, e):
    r = F12_ONE
    while e:
        if e & 1:
            r = f12_mul(r, a)
        a = f12_sqr(a)
        e >>= 1
    return r


# Frobenius: coefficients (u+1)^((p^n-1)/k)  (vendor/blst/src/fp12_tower.c:675-724)
def frob_coeffs(n):
    """gamma[i] = xi^(i*(p^n-1)/6) for i=0..5"""
    e = (P ** n - 1) // 6
    g = f2_pow(XI, e)
    out = [F2_ONE]
    for _ in range(5):
        out.append(f2_mul(out[-1], g))
    return out


_FROB = {n: frob_coeffs(n) for n in (1, 2, 3)}


def f12_frob(a, n=1):
    """a^(p^n).  Element = sum_{j,i} a[j][i] v^i w^j,  v^i w^j = w^(2i+j)."""
    g = _FROB[n]
    out = [[None] * 3, [None] * 3]
    for j in range(2):
        for i in range(3):
            c = a[j][i]
            if n & 1:
                c = f2_conj(c)
            out[j][i] = f2_mul(c, g[2 * i + j])
    return (tuple(out[0]), tuple(out[1]))


def f12_to_bytes(a):
    """blst_bendian_from_fp12 (vendor/blst/src/fp12_tower.c:773-786)."""
    out = b""
    for i in range(3):
        for j in range(2):
            out += a[j][i][0].to_bytes(48, "big") + a[j][i][1].to_bytes(48, "big")
    return out


def f12_from_bytes(b):
    a = [[None] * 3, [None] * 3]
    k = 0
    for i in range(3):
        for j in range(2):
            a[j][i] = (int.from_bytes(b[k:k + 48], "big"), int.from_bytes(b[k + 48:k + 96], "big"))
            k += 96
    return (tuple(a[0]), tuple(a[1]))


# ----------------------------------------------------------------------------
# curves.  G1: y^2 = x^3 + 4 over Fp (affine tuples or None = infinity)
G1_GEN = (
    0x17f1d3a73197d7942695638c4fa9ac0fc3688c4f9774b905a14e3a3f171bac586c55e83ff97a1aeffb3af00adb22c6bb,
    0x08b3f481e3aaa0f1a09e30ed741d8ae4fcf5e095d5d00af600db18cb2c04b3edd03cc744a2888ae40caa232946c5e7e1,
)
G2_GEN = (
    (0x024aa2b2f08f0a91260805272dc51051c6e47ad4fa403b02b4510b647ae3d1770bac0326a805bbefd48056c8c121bdb8,
     0x13e02b6052719f607dacd3a088274f65596bd0d09920b61ab5da61bbdc7f5049334cf11213945d57e5ac7d055d042b7e),
    (0x0ce5d527727d6e118cc9cdc6da2e351aadfd9baa8cbdd3a76d429a695160d12c923ac9cc3baca289e193548608b82801,
     0x0606c4a02ea734cc32acd2b02bc28b99cb3e287e85a763af267492ab572e99ab3f370d275cec1da1aaa9075ff05f79be),
)
B1 = 4
B2 = (4, 4)


def g1_add(p, q):
    if p is None:
        return q
    if q is None:
        return p
    if p[0] == q[0]:
        if (p[1] + q[1]) % P == 0:
            return None
        lam = 3 * p[0] * p[0] * inv(2 * p[1]) % P
    else:
        lam = (q[1] - p[1]) * inv(q[0] - p[0]) % P
    x = (lam * lam - p[0] - q[0]) % P
    return (x, (lam * (p[0] - x) - p[1]) % P)


def g1_neg(p):
    return None if p is None else (p[0], (-p[1]) % P)


def g1_mul(p, k):
    r = None
    while k:
        if k & 1:
            r = g1_add(r, p)
        p = g1_add(p, p)
        k >>= 1
    return r


def g2_add(p, q, a=F2_ZERO):
    """Affine addition on y^2 = x^3 + a x + b over Fp2 (a=0: E2; a=240i: E2')."""
    if p is None:
        return q
    if q is None:
        return p
    if p[0] == q[0]:
        if f2_add(p[1], q[1]) == F2_ZERO:
            return None
        lam = f2_mul(f2_add(f2_muli(f2_sqr(p[0]), 3), a), f2_inv(f2_muli(p[1], 2)))
    else:
        lam = f2_mul(f2_sub(q[1], p[1]), f2_inv(f2_sub(q[0], p[0])))
    x = f2_sub(f2_sub(f2_sqr(lam), p[0]), q[0])
    return (x, f2_sub(f2_mul(lam, f2_sub(p[0], x)), p[1]))


def g2_neg(p):
    return None if p is None else (p[0], f2_neg(p[1]))


def g2_mul(p, k):
    if k < 0:
        return g2_mul(g2_neg(p), -k)
    r = None
    while k:
        if k & 1:
            r = g2_add(r, p)
        p = g2_add(p, p)
        k >>= 1
    return r


def g1_on_curve(p):
    return p is None or (p[1] * p[1] - p[0] ** 3 - B1) % P == 0


def g2_on_curve(p):
    return p is None or f2_sub(f2_sqr(p[1]), f2_add(f2_mul(f2_sqr(p[0]), p[0]), B2)) == F2_ZERO


# psi endomorphism (vendor/blst/src/e2.c:455-482)
PSI_CX = f2_inv(f2_pow(XI, (P - 1) // 3))
PSI_CY = f2_inv(f2_pow(XI, (P - 1) // 2))


def g2_psi(p):
    if p is None:
        return None
    return (f2_mul(f2_conj(p[0]), PSI_CX), f2_mul(f2_conj(p[1]), PSI_CY))


def g2_clear_cofactor(p):
    """h_eff * P = [x^2-x-1]P + [x-1]psi(P) + psi^2(2P)  (map_to_g2.c:327-349; RFC 9380 G.4)."""
    t1 = g2_mul(p, X)
    t2 = g2_psi(p)
    t3 = g2_psi(g2_psi(g2_add(p, p)))
    t3 = g2_add(t3, g2_neg(t2))
    t2 = g2_add(t1, t2)
    t2 = g2_mul(t2, X)
    t3 = g2_add(t3, t2)
    t3 = g2_add(t3, g2_neg(t1))
    return g2_add(t3, g2_neg(p))


# ----------------------------------------------------------------------------
# serialisation (Zcash format; vendor/blst/src/e2.c:176-253, e1.c)
def g1_compress(p):
    if p is None:
        return bytes([0xc0]) + bytes(47)
    b = bytearray(p[0].to_bytes(48, "big"))
    b[0] |= 0x80
    if p[1] > (P - 1) // 2:
        b[0] |= 0x20
    return bytes(b)


def g1_serialize(p):
    if p is None:
        return bytes([0x40]) + bytes(95)
    return p[0].to_bytes(48, "big") + p[1].to_bytes(48, "big")


def g2_compress(p):
    if p is None:
        return bytes([0xc0]) + bytes(95)
    b = bytearray(p[0][1].to_bytes(48, "big") + p[0][0].to_bytes(48, "big"))
    b[0] |= 0x80
    y = p[1]
    big = (y[1] > (P - 1) // 2) if y[1] != 0 else (y[0] > (P - 1) // 2)
    if big:
        b[0] |= 0x20
    return bytes(b)


def g2_serialize(p):
    if p is None:
        return bytes([0x40]) + bytes(191)
    return (p[0][1].to_bytes(48, "big") + p[0][0].to_bytes(48, "big")
            + p[1][1].to_bytes(48, "big") + p[1][0].to_bytes(48, "big"))


def g1_uncompress(b):
    if b[0] & 0x40:
        return None
    x = int.from_bytes(bytes([b[0] & 0x1f]) + b[1:], "big")
    y = fp_sqrt((x ** 3 + 4) % P)
    if (y > (P - 1) // 2) != bool(b[0] & 0x20):
        y = P - y
    return (x, y)


# in-memory layout of the reference (blst_p1_affine/blst_p2_affine: LE limbs, Montgomery form)
def fp_to_mont_bytes(a):
    return (a * MONT_R % P).to_bytes(48, "little")


def fp_from_mont_bytes(b):
    return int.from_bytes(b, "little") * inv(MONT_R) % P


def g1_to_mem(p):
    if p is None:
        return bytes(96)
    return fp_to_mont_bytes(p[0]) + fp_to_mont_bytes(p[1])


def g1_from_mem(b):
    if b == bytes(96):
        return None
    return (fp_from_mont_bytes(b[:48]), fp_from_mont_bytes(b[48:96]))


def g2_to_mem(p):
    if p is None:
        return bytes(192)
    return b"".join(fp_to_mont_bytes(c) for c in (p[0][0], p[0][1], p[1][0], p[1][1]))


def g2_from_mem(b):
    if b == bytes(192):
        return None
    c = [fp_from_mont_bytes(b[i * 48:(i + 1) * 48]) for i in range(4)]
    return ((c[0], c[1]), (c[2], c[3]))


# ----------------------------------------------------------------------------
# hash to G2
def expand_message_xmd(msg, dst, len_in_bytes):
    """RFC 9380 5.3.1 with SHA-256 (vendor/blst/src/hash_to_field.c:51-114)."""
    if len(dst) > 255:
        dst = hashlib.sha256(b"H2C-OVERSIZE-DST-" + dst).digest()
    ell = (len_in_bytes + 31) // 32
    dst_prime = dst + bytes([len(dst)])
    b0 = hashlib.sha256(bytes(64) + msg + len_in_bytes.to_bytes(2, "big") + b"\x00" + dst_prime).digest()
    b = [hashlib.sha256(b0 + b"\x01" + dst_prime).digest()]
    for i in range(2, ell + 1):
        b.append(hashlib.sha256(bytes(x ^ y for x, y in zip(b0, b[-1])) + bytes([i]) + dst_prime).digest())
    return b"".join(b)[:len_in_bytes]


def hash_to_field_fp2(msg, dst, count=2):
    """vendor/blst/src/hash_to_field.c:120-154 ; order u0.re,u0.im,u1.re,u1.im"""
    L = 64
    u = expand_message_xmd(msg, dst, count * 2 * L)
    out = []
    for i in range(count):
        e = [int.from_bytes(u[L * (2 * i + j):L * (2 * i + j + 1)], "big") % P for j in range(2)]
        out.append((e[0], e[1]))
    return out


# SSWU on E2': y^2 = x^3 + 240i x + 1012(1+i)  (map_to_g2.c:13-26), Z = -(2+i) (:181-188)
SSWU_A = (0, 240)
SSWU_B = (1012, 1012)
SSWU_Z = ((-2) % P, (-1) % P)


def sswu_g2(u):
    """RFC 9380 6.6.2 map_to_curve_simple_swu, affine output on E2'."""
    A, B, Zc = SSWU_A, SSWU_B, SSWU_Z
    zu2 = f2_mul(Zc, f2_sqr(u))
    tv1 = f2_add(f2_sqr(zu2), zu2)
    if tv1 == F2_ZERO:
        x1 = f2_mul(B, f2_inv(f2_mul(Zc, A)))
    else:
        x1 = f2_mul(f2_mul(f2_neg(B), f2_inv(A)), f2_add(F2_ONE, f2_inv(tv1)))
    gx1 = f2_add(f2_add(f2_mul(f2_sqr(x1), x1), f2_mul(A, x1)), B)
    x2 = f2_mul(zu2, x1)
    gx2 = f2_add(f2_add(f2_mul(f2_sqr(x2), x2), f2_mul(A, x2)), B)
    if f2_is_square(gx1):
        x, y = x1, f2_sqrt(gx1)
    else:
        x, y = x2, f2_sqrt(gx2)
    if f2_sgn0(u) != f2_sgn0(y):
        y = f2_neg(y)
    return (x, y)


# 3-isogeny E2' -> E2, RFC 9380 appendix E.3 (map_to_g2.c:50-134 holds the same values in Montgomery form)
_K = 0x5c759507e8e333ebb5b7a9a47d7ed8532c52d39fd3a042a88b58423c50ae15d5c2638e343d9c71c6238aaaaaaaa97d6
ISO3_XNUM = [
    (_K, _K),
    (0, 0x11560bf17baa99bc32126fced787c88f984f87adf7ae0c7f9a208c6b4f20a4181472aaa9cb8d555526a9ffffffffc71a),
    (0x11560bf17baa99bc32126fced787c88f984f87adf7ae0c7f9a208c6b4f20a4181472aaa9cb8d555526a9ffffffffc71e,
     0x8ab05f8bdd54cde190937e76bc3e447cc27c3d6fbd7063fcd104635a790520c0a395554e5c6aaaa9354ffffffffe38d),
    (0x171d6541fa38ccfaed6dea691f5fb614cb14b4e7f4e810aa22d6108f142b85757098e38d0f671c7188e2aaaaaaaa5ed1, 0),
]
ISO3_XDEN = [
    (0, 0x1a0111ea397fe69a4b1ba7b6434bacd764774b84f38512bf6730d2a0f6b0f6241eabfffeb153ffffb9feffffffffaa63),
    (0xc, 0x1a0111ea397fe69a4b1ba7b6434bacd764774b84f38512bf6730d2a0f6b0f6241eabfffeb153ffffb9feffffffffaa9f),
    (1, 0),
]
ISO3_YNUM = [
    (0x1530477c7ab4113b59a4c18b076d11930f7da5d4a07f649bf54439d87d27e500fc8c25ebf8c92f6812cfc71c71c6d706,
     0x1530477c7ab4113b59a4c18b076d11930f7da5d4a07f649bf54439d87d27e500fc8c25ebf8c92f6812cfc71c71c6d706),
    (0, 0x5c759507e8e333ebb5b7a9a47d7ed8532c52d39fd3a042a88b58423c50ae15d5c2638e343d9c71c6238aaaaaaaa97be),
    (0x11560bf17baa99bc32126fced787c88f984f87adf7ae0c7f9a208c6b4f20a4181472aaa9cb8d555526a9ffffffffc71c,
     0x8ab05f8bdd54cde190937e76bc3e447cc27c3d6fbd7063fcd104635a790520c0a395554e5c6aaaa9354ffffffffe38f),
    (0x124c9ad43b6cf79bfbf7043de3811ad0761b0f37a1e26286b0e977c69aa274524e79097a56dc4bd9e1b371c71c718b10, 0),
]
ISO3_YDEN = [
    (0x1a0111ea397fe69a4b1ba7b6434bacd764774b84f38512bf6730d2a0f6b0f6241eabfffeb153ffffb9feffffffffa8fb,
     0x1a0111ea397fe69a4b1ba7b6434bacd764774b84f38512bf6730d2a0f6b0f6241eabfffeb153ffffb9feffffffffa8fb),
    (0, 0x1a0111ea397fe69a4b1ba7b6434bacd764774b84f38512bf6730d2a0f6b0f6241eabfffeb153ffffb9feffffffffa9d3),
    (0x12, 0x1a0111ea397fe69a4b1ba7b6434bacd764774b84f38512bf6730d2a0f6b0f6241eabfffeb153ffffb9feffffffffaa99),
    (1, 0),
]


def _horner(coeffs, x):
    r = F2_ZERO
    for c in reversed(coeffs):
        r = f2_add(f2_mul(r, x), c)
    return r


def iso3_g2(p):
    if p is None:
        return None
    x, y = p
    xn, xd = _horner(ISO3_XNUM, x), _horner(ISO3_XDEN, x)
    yn, yd = _horner(ISO3_YNUM, x), _horner(ISO3_YDEN, x)
    if xd == F2_ZERO or yd == F2_ZERO:
        return None
    return (f2_mul(xn, f2_inv(xd)), f2_mul(y, f2_mul(yn, f2_inv(yd))))


def hash_to_g2(msg, dst=DST_ETH2):
    """Hash_to_G2 (map_to_g2.c:388-396) with aug=""; returns affine point."""
    u0, u1 = hash_to_field_fp2(msg, dst, 2)
    q = g2_add(sswu_g2(u0), sswu_g2(u1), a=SSWU_A)
    return g2_clear_cofactor(iso3_g2(q))


# ----------------------------------------------------------------------------
# pairing: textbook Miller loop on the untwisted point, f_{|x|,Q}(P) conjugated (x<0)
def _embed_fp(a):
    return (((a % P, 0), F2_ZERO, F2_ZERO), F6_ZERO)


def _line_sparse(l0, l1, l2):
    """'xy00z0' layout: a[0][0]=l0, a[0][1]=l1, a[1][1]=l2 (pairing.c:155, :187-191)."""
    return ((l0, l1, F2_ZERO), (F2_ZERO, l2, F2_ZERO))


def miller_loop(Pp, Q):
    """f_{|x|,Q}(P) up to factors killed by the final exponentiation, conjugated.

    Line through T (slope lam, twist coordinates) evaluated at P and scaled by w^3:
        l = (lam*xT - yT) + (-lam*xP) * v + yP * v*w
    """
    if Pp is None or Q is None:
        return F12_ONE
    xp, yp = Pp
    f = F12_ONE
    T = Q
    bits = bin(Z_ABS)[3:]
    for b in bits:
        lam = f2_mul(f2_muli(f2_sqr(T[0]), 3), f2_inv(f2_muli(T[1], 2)))
        line = _line_sparse(f2_sub(f2_mul(lam, T[0]), T[1]), f2_muli(f2_neg(lam), xp), (yp, 0))
        f = f12_mul(f12_sqr(f), line)
        T = g2_add(T, T)
        if b == "1":
            lam = f2_mul(f2_sub(Q[1], T[1]), f2_inv(f2_sub(Q[0], T[0])))
            line = _line_sparse(f2_sub(f2_mul(lam, T[0]), T[1]), f2_muli(f2_neg(lam), xp), (yp, 0))
            f = f12_mul(f, line)
            T = g2_add(T, Q)
    return f12_conj(f)


FINAL_EXP_POWER = 3 * (P ** 12 - 1) // R_ORDER
HARD_POWER = 3 * (P ** 4 - P ** 2 + 1) // R_ORDER
assert HARD_POWER == (X - 1) ** 2 * (X + P) * (X * X + P * P - 1) + 3


def _cyc_exp_x(a):
    """a^x for a in the cyclotomic subgroup (x negative)."""
    return f12_conj(f12_pow(a, Z_ABS))


def final_exp(f):
    """f^(3*(p^12-1)/r)  (pairing.c:371-404)."""
    # easy part: (p^6-1)(p^2+1)
    t = f12_mul(f12_conj(f), f12_inv(f))
    t = f12_mul(f12_frob(t, 2), t)
    # hard part: (x-1)^2 (x+p) (x^2+p^2-1) + 3
    a = f12_mul(_cyc_exp_x(t), f12_conj(t))
    a = f12_mul(_cyc_exp_x(a), f12_conj(a))
    b = f12_mul(_cyc_exp_x(a), f12_frob(a, 1))
    c = f12_mul(f12_mul(_cyc_exp_x(_cyc_exp_x(b)), f12_frob(b, 2)), f12_conj(b))
    return f12_mul(c, f12_mul(f12_sqr(t), t))


# ----------------------------------------------------------------------------
# Nim layer: RLC scalars, chunking, batch verification
def parallel_chunks(num_chunks, total, cid):
    """blscurve/parallel_chunks.nim:42-55 -> (offset, size)."""
    base, rem = divmod(total, num_chunks)
    if cid < rem:
        return (base + 1) * cid, base + 1
    return base * cid + rem, base


def rlc_scalars(srb, n, chunks=0):
    """Per-set 64-bit blinding scalars.

    chunks == 0: serial mode, seed = SHA256(srb)          (blst_min_pubkey_sig_core.nim:502-505)
    chunks  > 0: parallel mode with numBatches = min(n, chunks); seed_c = SHA256(srb || LE64(c))
                 (bls_batch_verifier.nim:316, :333-336); per set seed <- SHA256(seed) until
                 LE64(seed[0:8]) != 0 (:551-554).
    """
    out = [0] * n
    if chunks == 0:
        ranges = [(hashlib.sha256(srb).digest(), 0, n)]
    else:
        nb = min(n, chunks)
        ranges = []
        for c in range(nb):
            off, sz = parallel_chunks(nb, n, c)
            ranges.append((hashlib.sha256(srb + c.to_bytes(8, "little")).digest(), off, sz))
    for seed, off, sz in ranges:
        for i in range(off, off + sz):
            seed = hashlib.sha256(seed).digest()
            while int.from_bytes(seed[:8], "little") == 0:
                seed = hashlib.sha256(seed).digest()
            out[i] = int.from_bytes(seed[:8], "little")
    return out


def combine_scalars(srb, n):
    """The n 64-bit scalars of MultiSignatureSet.combine (blst_min_pubkey_sig_core.nim:570-647): seed <- SHA256(seed)
    whenever the four little-endian 64-bit words of the current seed are used up, taken from the last word down; zero
    words are skipped."""
    seed, avail, sc = srb, 0, []
    while len(sc) < n:
        if avail == 0:
            seed, avail = hashlib.sha256(seed).digest(), 4
        avail -= 1
        v = int.from_bytes(seed[8 * avail:8 * avail + 8], "little")
        if v:
            sc.append(v)
    return sc


def batch_verify(sets, srb, chunks=0, scalars=None):
    """sets: list of (pk affine|None, msg bytes, sig affine|None).  Returns (ok, gt_bytes|None).

    Restates batchVerifySerial / batchVerifyParallel + aggregate.c:241-339, :460-501.
    """
    n = len(sets)
    if n == 0:
        return False, None
    if scalars is None:
        scalars = rlc_scalars(srb, n, chunks)
    S = None
    gt = F12_ONE
    for (pk, msg, sig), r in zip(sets, scalars):
        if sig is not None:
            S = g2_add(S, g2_mul(sig, r))
        if pk is None:
            return False, None
        gt = f12_mul(gt, miller_loop(g1_mul(pk, r), hash_to_g2(msg)))
    any_sig = any(s[2] is not None for s in sets)
    gtsig = miller_loop(G1_GEN, S) if any_sig else F12_ONE
    out = final_exp(f12_mul(f12_conj(gtsig), gt))
    return out == F12_ONE, f12_to_bytes(out)


# ----------------------------------------------------------------------------
# PublicKey / Signature fromBytes (bls_sig_io.nim:42-122 over blst_p1/p2_uncompress and _deserialize, e1.c / e2.c):
# returns (BLST_ERROR, affine point in memory layout, all zero on error).
#   0 SUCCESS, 1 BAD_ENCODING, 2 POINT_NOT_ON_CURVE, 3 POINT_NOT_IN_GROUP, 6 PK_IS_INFINITY
def _fp_from_be48(b, flags):
    v = int.from_bytes((bytes([b[0] & 0x1f]) + b[1:48]) if flags else b[:48], "big")
    return v if v < P else None


def _f2_largest(y):
    return y[1] > (P - 1) // 2 if y[1] else y[0] > (P - 1) // 2


def _point_from_bytes(raw, g2):
    size = 96 if g2 else 48                                   # compressed length
    b0 = raw[0]
    if len(raw) == 2 * size and b0 & 0xe0 == 0:               # uncompressed x || y
        c = [_fp_from_be48(raw[48 * k:48 * k + 48], k == 0) for k in range(len(raw) // 48)]
        if None in c:
            return 1, None
        pt = ((c[1], c[0]), (c[3], c[2])) if g2 else (c[0], c[1])
        if not (g2_on_curve(pt) if g2 else g1_on_curve(pt)):
            return 2, None
        return (3 if not g2 and pt[0] == 0 else 0), pt
    if b0 & 0x80:
        if b0 & 0x40:
            return (0 if b0 & 0x3f == 0 and not any(raw[1:size]) else 1), None
        if g2:
            c1, c0 = _fp_from_be48(raw[:48], True), _fp_from_be48(raw[48:96], False)
            if c1 is None or c0 is None:
                return 1, None
            x = (c0, c1)
            y = f2_sqrt(f2_add(f2_mul(f2_sqr(x), x), B2))
            if y is None:
                return 2, None
            if _f2_largest(y) != bool(b0 & 0x20):
                y = f2_neg(y)
            return 0, (x, y)
        x = _fp_from_be48(raw[:48], True)
        if x is None:
            return 1, None
        y = fp_sqrt((x ** 3 + B1) % P)
        if y is None:
            return 2, None
        if (y > (P - 1) // 2) != bool(b0 & 0x20):
            y = (P - y) % P
        return (3 if x == 0 else 0), (x, y)
    if len(raw) == 2 * size and b0 & 0x40 and b0 & 0x3f == 0 and not any(raw[1:]):
        return 0, None
    return 1, None


def pubkey_from_bytes(raw, group_check=True):
    err, pt = _point_from_bytes(raw, False)
    if err == 0 and pt is None:
        err = 6
    if err == 0 and group_check and g1_mul(pt, R_ORDER) is not None:
        err = 3
    return err, g1_to_mem(pt if err == 0 else None)


def signature_from_bytes(raw, group_check=True):
    err, pt = _point_from_bytes(raw, True)
    if err == 0 and group_check and g2_mul(pt, R_ORDER) is not None:
        err = 3
    return err, g2_to_mem(pt if err == 0 else None)
