// ec.cuh — short-Weierstrass point arithmetic (a = 0) over Fp (G1) and Fp2 (G2), Jacobian coordinates.
//
// Restates the *results* of vendor/blst/src/ec_ops.h (POINT_DADD_IMPL :40, POINT_DADD_AFFINE_IMPL_A0
// :129, POINT_DOUBLE_IMPL_A0 :299), ec_mult.h:178-223 (64-bit scalar multiplication) and
// e1.c:60-75 / e2.c:97-112 (to affine).  Formulas are the textbook dbl-2009-l / add-2007-bl /
// madd-2007-bl with explicit handling of infinity, P == Q and P == -Q; all outputs that leave the
// device are affine, hence canonical and comparable bit-for-bit with BLST.
// Conventions as in the reference: affine infinity = all-zero (x, y); Jacobian infinity = Z == 0.
#pragma once
#include "fpx.cuh"

namespace bls {

// ---- uniform field interface for the templates -------------------------------------------------
BLS_FN void f_add(fp &r, const fp &a, const fp &b) { fp_add(r, a, b); }
BLS_FN void f_sub(fp &r, const fp &a, const fp &b) { fp_sub(r, a, b); }
BLS_FN void f_dbl(fp &r, const fp &a) { fp_dbl(r, a); }
BLS_FN void f_neg(fp &r, const fp &a) { fp_neg(r, a); }
BLS_FN void f_mul(fp &r, const fp &a, const fp &b) { fp_mul_ni(r, a, b); }
BLS_FN void f_sqr(fp &r, const fp &a) { fp_sqr_ni(r, a); }
BLS_FN bool f_is_zero(const fp &a) { return fp_is_zero(a); }
BLS_FN bool f_eq(const fp &a, const fp &b) { return fp_eq(a, b); }
BLS_FN void f_set_zero(fp &r) { fp_set_zero(r); }
BLS_FN void f_set_one(fp &r) { r = FP_ONE; }
BLS_FN void f_inv(fp &r, const fp &a) { fp_inv(r, a); }

BLS_FN void f_add(fp2 &r, const fp2 &a, const fp2 &b) { fp2_add(r, a, b); }
BLS_FN void f_sub(fp2 &r, const fp2 &a, const fp2 &b) { fp2_sub(r, a, b); }
BLS_FN void f_dbl(fp2 &r, const fp2 &a) { fp2_dbl(r, a); }
BLS_FN void f_neg(fp2 &r, const fp2 &a) { fp2_neg(r, a); }
BLS_FN void f_mul(fp2 &r, const fp2 &a, const fp2 &b) { fp2_mul(r, a, b); }
BLS_FN void f_sqr(fp2 &r, const fp2 &a) { fp2_sqr(r, a); }
BLS_FN bool f_is_zero(const fp2 &a) { return fp2_is_zero(a); }
BLS_FN bool f_eq(const fp2 &a, const fp2 &b) { return fp2_eq(a, b); }
BLS_FN void f_set_zero(fp2 &r) { fp2_set_zero(r); }
BLS_FN void f_set_one(fp2 &r) { r.c0 = FP_ONE; fp_set_zero(r.c1); }
BLS_FN void f_inv(fp2 &r, const fp2 &a) { fp2_inv(r, a); }
BLS_FN void f_inv_vt(fp &r, const fp &a) { fp_inv_vartime(r, a); }
BLS_FN void f_inv_vt(fp2 &r, const fp2 &a) { fp2_inv_vartime(r, a); }

template <class F> struct jac_t { F x, y, z; };
template <class F> struct aff_t { F x, y; };
typedef jac_t<fp> g1_jac;
typedef aff_t<fp> g1_aff;
typedef jac_t<fp2> g2_jac;
typedef aff_t<fp2> g2_aff;

template <class F> BLS_FN bool pt_is_inf(const jac_t<F> &p) { return f_is_zero(p.z); }
template <class F> BLS_FN bool aff_is_inf(const aff_t<F> &p) { return f_is_zero(p.x) & f_is_zero(p.y); }
template <class F> BLS_FN void pt_set_inf(jac_t<F> &p) { f_set_zero(p.x); f_set_zero(p.y); f_set_zero(p.z); }
template <class F> BLS_FN void pt_from_affine(jac_t<F> &r, const aff_t<F> &a) {
    r.x = a.x;
    r.y = a.y;
    if (aff_is_inf(a)) f_set_zero(r.z); else f_set_one(r.z);
}
template <class F> BLS_FN void pt_neg(jac_t<F> &r, const jac_t<F> &a) { r.x = a.x; f_neg(r.y, a.y); r.z = a.z; }

// dbl-2009-l (a = 0): 2M + 5S.  Infinity (Z=0) and order-2 points (Y=0) map to Z3 = 0.
template <class F> BLS_NOINLINE void pt_dbl(jac_t<F> &r, const jac_t<F> &p) {
    F A, B, C, D, E, Fq, t;
    f_sqr(A, p.x);
    f_sqr(B, p.y);
    f_sqr(C, B);
    f_add(t, p.x, B);
    f_sqr(t, t);
    f_sub(t, t, A);
    f_sub(t, t, C);
    f_dbl(D, t);                 // D = 2((X+B)^2 - A - C)
    f_dbl(E, A);
    f_add(E, E, A);              // E = 3A
    f_sqr(Fq, E);
    f_mul(t, p.y, p.z);
    f_dbl(r.z, t);               // Z3 = 2YZ   (before x,y are overwritten: r may alias p)
    f_sub(Fq, Fq, D);
    f_sub(Fq, Fq, D);            // X3 = F - 2D
    f_sub(t, D, Fq);
    f_mul(t, E, t);
    f_dbl(C, C);
    f_dbl(C, C);
    f_dbl(C, C);                 // 8C
    r.x = Fq;
    f_sub(r.y, t, C);
}

// general doubling with curve coefficient a (dbl-2007-bl); only used for the E2' corner case
template <class F> BLS_NOINLINE void pt_dbl_a(jac_t<F> &r, const jac_t<F> &p, const F &a) {
    F XX, YY, YYYY, ZZ, S, M, T, t;
    f_sqr(XX, p.x);
    f_sqr(YY, p.y);
    f_sqr(YYYY, YY);
    f_sqr(ZZ, p.z);
    f_add(t, p.x, YY);
    f_sqr(t, t);
    f_sub(t, t, XX);
    f_sub(t, t, YYYY);
    f_dbl(S, t);
    f_sqr(t, ZZ);
    f_mul(t, a, t);
    f_dbl(M, XX);
    f_add(M, M, XX);
    f_add(M, M, t);
    f_sqr(T, M);
    f_sub(T, T, S);
    f_sub(T, T, S);
    f_add(t, p.y, p.z);
    f_sqr(t, t);
    f_sub(t, t, YY);
    f_sub(r.z, t, ZZ);
    r.x = T;
    f_sub(t, S, T);
    f_mul(t, M, t);
    f_dbl(YYYY, YYYY);
    f_dbl(YYYY, YYYY);
    f_dbl(YYYY, YYYY);
    f_sub(r.y, t, YYYY);
}

// add-2007-bl: 11M + 5S, complete by case analysis.  `a_coeff` (nullable) is only consulted when
// the inputs turn out to be equal and the curve is not a=0 (hash-to-curve adds on E2').
template <class F> BLS_NOINLINE void pt_add(jac_t<F> &r, const jac_t<F> &p, const jac_t<F> &q, const F *a_coeff = nullptr) {
    if (pt_is_inf(p)) { r = q; return; }
    if (pt_is_inf(q)) { r = p; return; }
    F Z1Z1, Z2Z2, U1, U2, S1, S2, H, I, J, rr, V, t;
    f_sqr(Z1Z1, p.z);
    f_sqr(Z2Z2, q.z);
    f_mul(U1, p.x, Z2Z2);
    f_mul(U2, q.x, Z1Z1);
    f_mul(t, q.z, Z2Z2);
    f_mul(S1, p.y, t);
    f_mul(t, p.z, Z1Z1);
    f_mul(S2, q.y, t);
    f_sub(H, U2, U1);
    f_sub(rr, S2, S1);
    if (f_is_zero(H)) {
        if (f_is_zero(rr)) {
            if (a_coeff) pt_dbl_a(r, p, *a_coeff); else pt_dbl(r, p);
        } else {
            pt_set_inf(r);
        }
        return;
    }
    f_dbl(rr, rr);
    f_dbl(I, H);
    f_sqr(I, I);
    f_mul(J, H, I);
    f_mul(V, U1, I);
    f_add(t, p.z, q.z);
    f_sqr(t, t);
    f_sub(t, t, Z1Z1);
    f_sub(t, t, Z2Z2);
    f_mul(r.z, t, H);
    f_sqr(t, rr);
    f_sub(t, t, J);
    f_sub(t, t, V);
    f_sub(t, t, V);              // X3
    r.x = t;
    f_sub(t, V, t);
    f_mul(t, rr, t);
    f_mul(S1, S1, J);
    f_dbl(S1, S1);
    f_sub(r.y, t, S1);
}

// madd-2007-bl: 7M + 4S, q affine (all-zero = infinity)
template <class F> BLS_NOINLINE void pt_add_affine(jac_t<F> &r, const jac_t<F> &p, const aff_t<F> &q) {
    if (aff_is_inf(q)) { r = p; return; }
    if (pt_is_inf(p)) { pt_from_affine(r, q); return; }
    F Z1Z1, U2, S2, H, HH, I, J, rr, V, t;
    f_sqr(Z1Z1, p.z);
    f_mul(U2, q.x, Z1Z1);
    f_mul(t, p.z, Z1Z1);
    f_mul(S2, q.y, t);
    f_sub(H, U2, p.x);
    f_sub(rr, S2, p.y);
    if (f_is_zero(H)) {
        if (f_is_zero(rr)) pt_dbl(r, p); else pt_set_inf(r);
        return;
    }
    f_dbl(rr, rr);
    f_sqr(HH, H);
    f_dbl(I, HH);
    f_dbl(I, I);
    f_mul(J, H, I);
    f_mul(V, p.x, I);
    f_add(t, p.z, H);
    f_sqr(t, t);
    f_sub(t, t, Z1Z1);
    F y1 = p.y;
    f_sub(r.z, t, HH);
    f_sqr(t, rr);
    f_sub(t, t, J);
    f_sub(t, t, V);
    f_sub(t, t, V);
    r.x = t;
    f_sub(t, V, t);
    f_mul(t, rr, t);
    f_mul(J, y1, J);
    f_dbl(J, J);
    f_sub(r.y, t, J);
}

// affine from Jacobian (infinity -> all zero)
template <class F> BLS_NOINLINE void pt_to_affine(aff_t<F> &r, const jac_t<F> &p) {
    if (pt_is_inf(p)) { f_set_zero(r.x); f_set_zero(r.y); return; }
    F zi, zi2;
    f_inv(zi, p.z);
    f_sqr(zi2, zi);
    f_mul(r.x, p.x, zi2);
    f_mul(zi2, zi2, zi);
    f_mul(r.y, p.y, zi2);
}

// same through the variable-time inversion: for kernels where ONE thread normalises one public point
template <class F> BLS_NOINLINE void pt_to_affine_vt(aff_t<F> &r, const jac_t<F> &p) {
    if (pt_is_inf(p)) { f_set_zero(r.x); f_set_zero(r.y); return; }
    F zi, zi2;
    f_inv_vt(zi, p.z);
    f_sqr(zi2, zi);
    f_mul(r.x, p.x, zi2);
    f_mul(zi2, zi2, zi);
    f_mul(r.y, p.y, zi2);
}

// same, with 1/Z supplied (batch inversion)
template <class F> BLS_NOINLINE void pt_to_affine_zinv(aff_t<F> &r, const jac_t<F> &p, const F &zi) {
    if (pt_is_inf(p)) { f_set_zero(r.x); f_set_zero(r.y); return; }
    F zi2;
    f_sqr(zi2, zi);
    f_mul(r.x, p.x, zi2);
    f_mul(zi2, zi2, zi);
    f_mul(r.y, p.y, zi2);
}

// Homogeneous (X : Y : Z), x = X / Z and y = Y / Z: the point form of the dataflow programs (fpprog.hpp), 3 F per point.
// from Jacobian: (X Z : Y : Z^3); infinity -> (0 : 1 : 0)
template <class F> BLS_NOINLINE void pt_jac_to_hom(F *h, const jac_t<F> &p) {
    F x, y, z;
    if (pt_is_inf(p)) {
        f_set_zero(x); f_set_one(y); f_set_zero(z);
    } else {
        F z2;
        f_mul(x, p.x, p.z);
        y = p.y;
        f_sqr(z2, p.z);
        f_mul(z, z2, p.z);
    }
    h[0] = x; h[1] = y; h[2] = z;
}

// to Jacobian (X Z, Y Z^2, Z); Z = 0 -> infinity
template <class F> BLS_FN void pt_hom_to_jac(jac_t<F> &r, const F *h) {
    const F X = h[0], Y = h[1], Z = h[2];
    if (f_is_zero(Z)) pt_set_inf(r);
    else { F z2; f_mul(r.x, X, Z); f_sqr(z2, Z); f_mul(r.y, Y, z2); r.z = Z; }
}

// to affine (X / Z, Y / Z) through the variable-time inversion; Z = 0 -> 0 -> the all-zero affine encoding of infinity
template <class F> BLS_FN void pt_hom_to_affine(aff_t<F> &r, const F *h) {
    const F X = h[0], Y = h[1], Z = h[2];
    F zi;
    f_inv_vt(zi, Z);
    f_mul(r.x, X, zi);
    f_mul(r.y, Y, zi);
}

// r = [k]P for a 64-bit k, P affine: MSB-first double-and-add with mixed additions.
// (BLST uses a 5-bit Booth window, ec_mult.h:178-223; the affine result is the same point.)
template <class F> BLS_NOINLINE void pt_mul_u64(jac_t<F> &r, const aff_t<F> &p, uint64_t k) {
    jac_t<F> acc;
    pt_set_inf(acc);
    if (k != 0 && !aff_is_inf(p)) {
        int top = 63;
        while (!((k >> top) & 1)) top--;
        pt_from_affine(acc, p);
        for (int i = top - 1; i >= 0; i--) {
            pt_dbl(acc, acc);
            if ((k >> i) & 1) pt_add_affine(acc, acc, p);
        }
    }
    r = acc;
}

// r = [k]P for a 64-bit k, P affine: signed 4-bit windows (digits in [-8, 8], 17 of them), 8-entry table.
// Every lane of a warp does the same 64 doublings + 17 additions whatever its scalar, where double-and-add under
// divergence pays 63 + 63; 781 instead of 1134 field multiplications in G1.  (BLST: 5-bit Booth, ec_mult.h:178-223.)
template <class F> BLS_NOINLINE void pt_mul_u64_w4(jac_t<F> &r, const aff_t<F> &p, uint64_t k) {
    jac_t<F> tbl[8], acc;                        // tbl[i] = [i+1]P
    pt_from_affine(tbl[0], p);
    pt_dbl(tbl[1], tbl[0]);
    pt_add_affine(tbl[2], tbl[1], p);
    pt_dbl(tbl[3], tbl[1]);
    pt_add_affine(tbl[4], tbl[3], p);
    pt_dbl(tbl[5], tbl[2]);
    pt_add_affine(tbl[6], tbl[5], p);
    pt_dbl(tbl[7], tbl[3]);
    int dig[17], carry = 0;
    for (int j = 0; j < 16; j++) {
        int w = (int)((k >> (4 * j)) & 15) + carry;
        if (w > 8) { w -= 16; carry = 1; } else carry = 0;
        dig[j] = w;
    }
    dig[16] = carry;
    pt_set_inf(acc);
    for (int j = 16; j >= 0; j--) {
        if (j != 16) for (int d = 0; d < 4; d++) pt_dbl(acc, acc);
        const int d = dig[j];
        if (d != 0) {
            jac_t<F> q = tbl[(d < 0 ? -d : d) - 1];
            if (d < 0) f_neg(q.y, q.y);
            pt_add(acc, acc, q);
        }
    }
    r = acc;
}

// r = [k]P, P Jacobian, k given as nwords little-endian u32 words (top bit need not be set)
template <class F> BLS_NOINLINE void pt_mul_words(jac_t<F> &r, const jac_t<F> &p, const uint32_t *k, int nwords) {
    jac_t<F> acc;
    pt_set_inf(acc);
    int i = nwords * 32 - 1;
    while (i >= 0 && !((k[i >> 5] >> (i & 31)) & 1)) i--;      // skip leading zero bits
    for (; i >= 0; i--) {
        pt_dbl(acc, acc);
        if ((k[i >> 5] >> (i & 31)) & 1) pt_add(acc, acc, p);
    }
    r = acc;
}

}  // namespace bls
