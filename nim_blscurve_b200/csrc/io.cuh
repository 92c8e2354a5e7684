// io.cuh — batched deserialisation with checks: wire bytes -> affine points in Montgomery form (SURVEY.md §8f N2).
//
// Restates the results of PublicKey.fromBytes / Signature.fromBytes (blscurve/blst/bls_sig_io.nim:42-122) over
//   blst_p1_uncompress  vendor/blst/src/e1.c:236-294      blst_p1_deserialize  e1.c:296-351
//   blst_p2_uncompress  vendor/blst/src/e2.c:279-343      blst_p2_deserialize  e2.c:345-410
//   blst_p1_affine_in_g1 e1.c:405-460                     blst_p2_affine_in_g2 map_to_g2.c:403-443
// including the BLST_ERROR each input earns (bindings/blst.h:47-56).  The arithmetic is this library's own:
// square roots are a^((p+1)/4) (Fp) and the complex method of fpx.cuh (Fp2); the subgroup tests are Scott's
// endomorphism equations — phi(P) = [-z^2]P on E1 and psi(P) = [z]P on E2 — which hold exactly on the order-r
// subgroups (M. Scott, "A note on group membership tests for G1, G2 and GT on BLS pairing-friendly curves"), where
// BLST uses a sigma-based chain for G1 (e1.c:405) and psi-based for G2; only the boolean is observable.
#pragma once
#include "h2c.cuh"

namespace bls {

enum { IO_SUCCESS = 0, IO_BAD_ENCODING = 1, IO_NOT_ON_CURVE = 2, IO_NOT_IN_GROUP = 3, IO_PK_IS_INFINITY = 6 };

// 48 big-endian bytes -> canonical limbs (top three bits cleared when mask_top); false when the value is >= p
BLS_FN bool fp_canon_from_be48(fp &r, const uint8_t *in, bool mask_top) {
    for (int k = 0; k < 12; k++) {
        const uint8_t *b = in + 44 - 4 * k;
        r.l[k] = ((uint32_t)b[0] << 24) | ((uint32_t)b[1] << 16) | ((uint32_t)b[2] << 8) | b[3];
    }
    if (mask_top) r.l[11] &= 0x1fffffffu;
    int64_t bw = 0;
    for (int i = 0; i < 12; i++) { bw += (int64_t)r.l[i] - P32(i); bw >>= 32; }
    return bw < 0;
}

BLS_FN void fp_to_mont(fp &r, const fp &canon) { fp_mul_ni(r, canon, FP_R2); }

// r = sqrt(a) when a is a square (returns true); p = 3 mod 4
BLS_NOINLINE bool fp_sqrt(fp &r, const fp &a) {
    fp t, s, chk;
    fp_pow_p34(t, a);                  // a^((p-3)/4)
    fp_mul_ni(s, t, a);                // a^((p+1)/4)
    fp_sqr_ni(chk, s);
    r = s;
    return fp_eq(chk, a);
}

BLS_NOINLINE bool fp2_sqrt(fp2 &r, const fp2 &a) {
    fp2 rs, s, chk;
    fp2_rsqrt_or_z(rs, a);             // 1/sqrt(a) when a is a square
    fp2_mul(s, a, rs);
    fp2_sqr(chk, s);
    r = s;
    return fp2_eq(chk, a);
}

BLS_FN bool fp_is_lexically_largest(const fp &a) {
    fp c;
    fp_from_mont(c, a);
    return fp_is_lexically_largest_canon(c);
}

// y^2 == x^3 + b
BLS_FN bool g1_on_curve(const g1_aff &p) {
    fp t, yy;
    fp_sqr_ni(t, p.x);
    fp_mul_ni(t, t, p.x);
    fp_add(t, t, G1_B);
    fp_sqr_ni(yy, p.y);
    return fp_eq(t, yy);
}
BLS_FN bool g2_on_curve(const g2_aff &p) {
    fp2 t, yy;
    fp2_sqr(t, p.x);
    fp2_mul(t, t, p.x);
    fp2_add(t, t, G2_B);
    fp2_sqr(yy, p.y);
    return fp2_eq(t, yy);
}

// [|z|]P on either curve: 63 doublings + 5 additions
template <class F> BLS_NOINLINE void pt_mul_by_zabs(jac_t<F> &r, const jac_t<F> &p) {
    jac_t<F> acc = p;
    const uint64_t z = BLS_Z_ABS;
    for (int i = 62; i >= 0; i--) {
        pt_dbl(acc, acc);
        if ((z >> i) & 1) pt_add(acc, acc, p);
    }
    r = acc;
}

// Jacobian T equals the affine point (x, y)?  (T at infinity never does)
template <class F> BLS_FN bool pt_eq_affine(const jac_t<F> &T, const F &x, const F &y) {
    if (pt_is_inf(T)) return false;
    F zz, zzz, l, rr;
    f_sqr(zz, T.z);
    f_mul(zzz, zz, T.z);
    f_mul(l, x, zz);
    f_mul(rr, y, zzz);
    return f_eq(l, T.x) & f_eq(rr, T.y);
}

// P in G1  <=>  [z^2]P == -phi(P) = (beta x, -y); infinity is in the group (blst_p1_affine_in_g1 on infinity: true)
BLS_NOINLINE bool g1_in_subgroup(const g1_aff &p) {
    if (aff_is_inf(p)) return true;
    g1_jac t;
    pt_from_affine(t, p);
    pt_mul_by_zabs(t, t);
    pt_mul_by_zabs(t, t);
    fp bx, ny;
    fp_mul_ni(bx, p.x, G1_BETA);
    fp_neg(ny, p.y);
    return pt_eq_affine(t, bx, ny);
}

// psi(P) == -T for the finite affine P and T = [|z|]P computed by the caller
BLS_FN bool g2_psi_is_neg(const g2_aff &p, const g2_jac &t) {
    g2_jac q;
    pt_from_affine(q, p);
    g2_psi(q, q);                      // affine in, Z stays 1
    fp2 ny;
    fp2_neg(ny, q.y);
    return pt_eq_affine(t, q.x, ny);
}

// P in G2  <=>  psi(P) == [z]P = -[|z|]P
BLS_NOINLINE bool g2_in_subgroup(const g2_aff &p) {
    if (aff_is_inf(p)) return true;
    g2_jac t, q;
    pt_from_affine(q, p);
    pt_mul_by_zabs(t, q);
    return g2_psi_is_neg(p, t);
}

// one compressed G1 point (48 bytes, flags already inspected by the caller: compressed, not infinity)
BLS_FN int g1_uncompress_body(g1_aff &out, const uint8_t *in) {
    fp xc, x, y;
    if (!fp_canon_from_be48(xc, in, true)) return IO_BAD_ENCODING;
    fp_to_mont(x, xc);
    fp t;
    fp_sqr_ni(t, x);
    fp_mul_ni(t, t, x);
    fp_add(t, t, G1_B);
    if (!fp_sqrt(y, t)) return IO_NOT_ON_CURVE;
    const bool want = (in[0] & 0x20) != 0;
    fp_cneg(y, y, fp_is_lexically_largest(y) != want);
    out.x = x;
    out.y = y;
    return fp_is_zero(x) ? IO_NOT_IN_GROUP : IO_SUCCESS;      // (0, +-2) has order 3
}

BLS_FN bool bytes_zero(const uint8_t *p, int n) {
    uint32_t acc = 0;
    for (int i = 0; i < n; i++) acc |= p[i];
    return acc == 0;
}

// blst_p1_uncompress (len 48) / blst_p1_deserialize (len 96)
BLS_NOINLINE int g1_from_bytes(g1_aff &out, const uint8_t *in, int len) {
    const uint8_t in0 = in[0];
    fp_set_zero(out.x);
    fp_set_zero(out.y);
    if (len == 96 && (in0 & 0xe0) == 0) {                    // uncompressed big-endian x || y
        fp xc, yc;
        if (!fp_canon_from_be48(xc, in, true)) return IO_BAD_ENCODING;
        if (!fp_canon_from_be48(yc, in + 48, false)) return IO_BAD_ENCODING;
        g1_aff p;
        fp_to_mont(p.x, xc);
        fp_to_mont(p.y, yc);
        if (!g1_on_curve(p)) return IO_NOT_ON_CURVE;
        out = p;
        return fp_is_zero(p.x) ? IO_NOT_IN_GROUP : IO_SUCCESS;
    }
    if (in0 & 0x80) {                                         // compressed
        if (in0 & 0x40) return ((in0 & 0x3f) == 0 && bytes_zero(in + 1, 47)) ? IO_SUCCESS : IO_BAD_ENCODING;
        return g1_uncompress_body(out, in);
    }
    if (len == 96 && (in0 & 0x40) && (in0 & 0x3f) == 0 && bytes_zero(in + 1, 95)) return IO_SUCCESS;   // infinity
    return IO_BAD_ENCODING;
}

BLS_FN int g2_uncompress_body(g2_aff &out, const uint8_t *in) {
    fp c1, c0;
    if (!fp_canon_from_be48(c1, in, true)) return IO_BAD_ENCODING;
    if (!fp_canon_from_be48(c0, in + 48, false)) return IO_BAD_ENCODING;
    fp2 x, y, t;
    fp_to_mont(x.c0, c0);
    fp_to_mont(x.c1, c1);
    fp2_sqr(t, x);
    fp2_mul(t, t, x);
    fp2_add(t, t, G2_B);
    if (!fp2_sqrt(y, t)) return IO_NOT_ON_CURVE;
    const bool want = (in[0] & 0x20) != 0;
    fp2_cneg(y, y, fp2_is_lexically_largest(y) != want);
    out.x = x;
    out.y = y;
    return IO_SUCCESS;
}

// blst_p2_uncompress (len 96) / blst_p2_deserialize (len 192)
BLS_NOINLINE int g2_from_bytes(g2_aff &out, const uint8_t *in, int len) {
    const uint8_t in0 = in[0];
    fp2_set_zero(out.x);
    fp2_set_zero(out.y);
    if (len == 192 && (in0 & 0xe0) == 0) {                   // x.im || x.re || y.im || y.re
        fp c[4];
        for (int k = 0; k < 4; k++)
            if (!fp_canon_from_be48(c[k], in + 48 * k, k == 0)) return IO_BAD_ENCODING;
        g2_aff p;
        fp_to_mont(p.x.c1, c[0]);
        fp_to_mont(p.x.c0, c[1]);
        fp_to_mont(p.y.c1, c[2]);
        fp_to_mont(p.y.c0, c[3]);
        if (!g2_on_curve(p)) return IO_NOT_ON_CURVE;
        out = p;
        return IO_SUCCESS;
    }
    if (in0 & 0x80) {
        if (in0 & 0x40) return ((in0 & 0x3f) == 0 && bytes_zero(in + 1, 95)) ? IO_SUCCESS : IO_BAD_ENCODING;
        return g2_uncompress_body(out, in);
    }
    if (len == 192 && (in0 & 0x40) && (in0 & 0x3f) == 0 && bytes_zero(in + 1, 191)) return IO_SUCCESS;
    return IO_BAD_ENCODING;
}

// PublicKey.fromBytes (bls_sig_io.nim:87-104): decode, reject infinity, subgroup check
BLS_FN int pubkey_from_bytes(g1_aff &out, const uint8_t *in, int len, bool group_check) {
    g1_aff p;
    int err = g1_from_bytes(p, in, len);
    if (err == IO_SUCCESS && aff_is_inf(p)) err = IO_PK_IS_INFINITY;
    if (err == IO_SUCCESS && group_check && !g1_in_subgroup(p)) err = IO_NOT_IN_GROUP;
    if (err != IO_SUCCESS) { fp_set_zero(p.x); fp_set_zero(p.y); }
    out = p;
    return err;
}

// Signature.fromBytes (bls_sig_io.nim:42-60): decode, subgroup check (infinity allowed)
BLS_FN int signature_from_bytes(g2_aff &out, const uint8_t *in, int len, bool group_check) {
    g2_aff p;
    int err = g2_from_bytes(p, in, len);
    if (err == IO_SUCCESS && group_check && !g2_in_subgroup(p)) err = IO_NOT_IN_GROUP;
    if (err != IO_SUCCESS) { fp2_set_zero(p.x); fp2_set_zero(p.y); }
    out = p;
    return err;
}

// Zcash compressed encoding of an affine G1 point (e1.c:208-234)
BLS_FN void g1_compress(uint8_t *out, const g1_aff &p) {
    if (aff_is_inf(p)) {
        out[0] = 0xc0;
        for (int i = 1; i < 48; i++) out[i] = 0;
        return;
    }
    fp c;
    fp_from_mont(c, p.x);
    for (int i = 0; i < 48; i++) out[i] = (uint8_t)(c.l[(47 - i) >> 2] >> (8 * ((47 - i) & 3)));
    out[0] |= 0x80;
    if (fp_is_lexically_largest(p.y)) out[0] |= 0x20;
}

}  // namespace bls
