// tests/hostsim/hostsim.cpp — TEST INFRASTRUCTURE ONLY.
// Compiles the device arithmetic headers as plain C++ (no __CUDACC__) so that the tower / curve /
// hash / pairing logic can be checked against the oracle on a machine without a GPU.  The PTX
// bodies of fp.cuh are replaced by the portable branch there; the PTX itself is checked on the GPU
// by tests/test_gpu_*.py.  Never linked into libblsgpu.so.
#include <stdint.h>
#include <stddef.h>
#include <string.h>
#include "../../nim_blscurve_b200/csrc/h2c.cuh"
#include "../../nim_blscurve_b200/csrc/pairing.cuh"
#include "../../nim_blscurve_b200/csrc/io.cuh"
#include "../../nim_blscurve_b200/csrc/fpprog.hpp"
#include "../../nim_blscurve_b200/csrc/fplin.cuh"
#include "../../nim_blscurve_b200/csrc/route.hpp"
using namespace bls;

// subtractAll as blsgpu.cu: subtract_all arranges it: pairwise tree over (elems..., -dst), negated root, to affine
template <class F> static void hs_subtract(aff_t<F> *dst, const aff_t<F> *p, size_t n) {
    size_t m = n + 1;
    jac_t<F> *J = new jac_t<F>[m];
    for (size_t i = 0; i < n; i++) pt_from_affine(J[i], p[i]);
    pt_from_affine(J[n], *dst);
    pt_neg(J[n], J[n]);
    for (size_t k = m; k > 1;) {
        size_t half = (k + 1) / 2;
        for (size_t i = 0; i + half < k; i++) pt_add(J[i], J[i], J[i + half]);
        k = half;
    }
    pt_neg(J[0], J[0]);
    pt_to_affine_vt(*dst, J[0]);
    delete[] J;
}

extern "C" {
void hs_fp_mul(const fp *a, const fp *b, fp *r) { fp_mul(*r, *a, *b); }
void hs_fp_add(const fp *a, const fp *b, fp *r) { fp_add(*r, *a, *b); }
void hs_fp_sub(const fp *a, const fp *b, fp *r) { fp_sub(*r, *a, *b); }
void hs_fp_inv(const fp *a, fp *r) { fp_inv(*r, *a); }
void hs_fp_inv_vartime(const fp *a, fp *r) { fp_inv_vartime(*r, *a); }
int hs_fp2_rsqrt(const fp2 *a, fp2 *r) { return fp2_rsqrt_or_z(*r, *a) ? 1 : 0; }
void hs_hash_to_g2(const uint8_t *msg, size_t len, const uint8_t *dst, uint32_t dst_len, g2_aff *aff, uint8_t *comp) {
    g2_jac j;
    hash_to_g2_jac(j, msg, len, dst, dst_len);
    pt_to_affine(*aff, j);
    g2_compress(comp, *aff);
}
void hs_g1_mul_u64(const g1_aff *p, uint64_t k, g1_aff *r) { g1_jac j; pt_mul_u64(j, *p, k); pt_to_affine(*r, j); }
void hs_g1_mul_u64_w4(const g1_aff *p, uint64_t k, g1_aff *r) { g1_jac j; pt_mul_u64_w4(j, *p, k); pt_to_affine(*r, j); }
void hs_g2_mul_u64(const g2_aff *p, uint64_t k, g2_aff *r) { g2_jac j; pt_mul_u64(j, *p, k); pt_to_affine(*r, j); }

void hs_fp12_mul(const fp12 *a, const fp12 *b, fp12 *r) { fp12_mul(*r, *a, *b); }
void hs_fp12_sqr(const fp12 *a, fp12 *r) { fp12_sqr(*r, *a); }
void hs_fp12_cyc_sqr(const fp12 *a, fp12 *r) { fp12_cyc_sqr(*r, *a); }
void hs_fp12_inv(const fp12 *a, fp12 *r) { fp12_inv(*r, *a); }
void hs_fp12_frob(const fp12 *a, int n, fp12 *r) { fp12_frob(*r, *a, n); }
void hs_fp12_bytes(const fp12 *a, uint8_t *out) { fp12_to_bytes(out, *a); }
void hs_fp12_mul_by_line(fp12 *f, const fp2 *l) { fp12_mul_by_line(*f, l[0], l[1], l[2]); }
void hs_miller_loop_n(const g2_aff *Q, const g1_aff *P, int n, fp12 *f) {
    g2_jac T[16]; fp npx[16];
    miller_loop_n(*f, Q, P, n, T, npx);
}
void hs_final_exp(const fp12 *f, fp12 *r) { final_exp(*r, *f); }

// whole batch-verification pipeline as the kernels of kernels.cuh sequence it, executed on the host
struct hs_sigset { g1_aff pk; uint8_t msg[32]; g2_aff sig; };
int hs_batch_verify(const hs_sigset *sets, size_t n, const uint64_t *r, int group, int nseg, uint8_t *gt_out) {
    static const uint8_t dst[] = "BLS_SIG_BLS12381G2_XMD:SHA-256_SSWU_RO_POP_";
    memset(gt_out, 0, 576);
    if (n == 0) return 0;
    const size_t np = n + 1;                       // + the signature-side pair (S, -G1)
    g2_aff *Q = new g2_aff[np];
    g1_aff *P = new g1_aff[np];
    g2_jac S; pt_set_inf(S);
    int pk_inf = 0;
    for (size_t i = 0; i < n; i++) {
        g2_jac h; hash_to_g2_jac(h, sets[i].msg, 32, dst, 43);
        if (aff_is_inf(sets[i].pk)) pk_inf = 1;
        g1_jac pj; pt_mul_u64_w4(pj, sets[i].pk, r[i]);
        pt_to_affine(Q[i], h);
        pt_to_affine(P[i], pj);
        g2_jac sj; pt_mul_u64(sj, sets[i].sig, r[i]);
        pt_add(S, S, sj);
    }
    pt_to_affine(Q[n], S);
    P[n].x = G1_GEN_X;
    fp_neg(P[n].y, G1_GEN_Y);
    // kernel L: lines of every pair, word-major over pairs
    const size_t stride = (np + 31) & ~(size_t)31;
    uint32_t *lines = new uint32_t[(size_t)ML_NLINES * ML_LINE_WORDS * stride];
    for (size_t p = 0; p < np; p++) miller_lines(Q[p], P[p], lines + p, stride);
    // kernel A + row products: one Fp12 per segment
    const size_t ngroups = (np + group - 1) / group;
    fp12 *seg = new fp12[nseg];
    for (int j = 0; j < nseg; j++) {
        fp12_set_one(seg[j]);
        for (size_t g = 0; g < ngroups; g++) {
            fp12 f;
            miller_accumulate(f, lines, stride, np, g, ngroups, group, ml_seg_hi(j, nseg), ml_seg_lo(j, nseg));
            fp12_mul(seg[j], seg[j], f);
        }
    }
    fp12 F, gt;
    miller_combine(F, seg, nseg);
    final_exp(gt, F);
    fp12_to_bytes(gt_out, gt);
    delete[] Q; delete[] P; delete[] lines; delete[] seg;
    if (pk_inf) { memset(gt_out, 0, 576); return 0; }
    return fp12_is_one(gt) ? 1 : 0;
}
void hs_aggregate_g1(const g1_aff *p, size_t n, g1_aff *out) {
    g1_jac acc; pt_from_affine(acc, p[0]);
    for (size_t i = 1; i < n; i++) { g1_jac t; pt_from_affine(t, p[i]); pt_add(acc, acc, t); }
    pt_to_affine(*out, acc);
}
void hs_aggregate_g2(const g2_aff *p, size_t n, g2_aff *out) {
    g2_jac acc; pt_from_affine(acc, p[0]);
    for (size_t i = 1; i < n; i++) { g2_jac t; pt_from_affine(t, p[i]); pt_add(acc, acc, t); }
    pt_to_affine(*out, acc);
}
void hs_subtract_g1(g1_aff *dst, const g1_aff *p, size_t n) { hs_subtract<fp>(dst, p, n); }
void hs_subtract_g2(g2_aff *dst, const g2_aff *p, size_t n) { hs_subtract<fp2>(dst, p, n); }

// ---- fpprog.hpp: execute a compiled tail program on the CPU exactly as k_fp_program does on the device ----
// format 2 (rounds of products and rounds of linear combinations), exactly as k_fp_program2 does on the device: the
// combinations go through the same lin_add_term / lin_finish of fplin.cuh
static void run_program2(const std::vector<uint32_t> &w, const fp *in0, const fp *in1, const fp *cst, fp *out0) {
    const uint32_t nr = w[0], nslots = w[1], nin = w[2], nout = w[3];
    std::vector<fp> slots(nslots);
    fp_set_zero(slots[0]);
    for (uint32_t e = 0; e < nin; e++) {
        uint32_t sl = w[4 + 2 * e], ref = w[5 + 2 * e], buf = ref >> 24, idx = ref & 0xffffffu;
        slots[sl] = (buf == 0 ? in0 : (buf == 1 ? in1 : cst))[idx];
    }
    const uint32_t *rp = w.data() + ((4 + 2 * (nin + nout) + 3) & ~3u);
    for (uint32_t r = 0; r < nr; r++, rp += 128) {
        fp res[32];
        bool wr[32];
        for (int l = 0; l < 32; l++) {              // all lanes read before any lane writes (stricter than the device)
            const uint32_t *x = rp + 4 * l;
            const uint32_t op = x[0] >> 30;
            wr[l] = false;
            if (op == 1) { fp_mul(res[l], slots[x[1] & 1023], slots[(x[1] >> 10) & 1023]); wr[l] = true; }
            else if (op == 2) {
                const uint32_t npos = (x[0] >> 17) & 7, nneg = (x[0] >> 14) & 7;
                const uint32_t t[7] = {x[1] & 0x3fffu, (x[1] >> 14) & 0x3fffu, x[2] & 0x3fffu, (x[2] >> 14) & 0x3fffu,
                                       x[3] & 0x3fffu, (x[3] >> 14) & 0x3fffu, x[0] & 0x3fffu};
                lin_acc A;
                lin_clear(A);
                for (uint32_t j = 0; j < npos; j++) lin_add_term(A.P, slots[t[j] & 1023], t[j] >> 10);
                for (uint32_t j = 0; j < nneg; j++) lin_add_term(A.N, slots[t[6 - j] & 1023], t[6 - j] >> 10);
                lin_finish(res[l], A);
                wr[l] = true;
            } else if (x[0]) out0[x[2]] = slots[x[1]];                                  // STORE
        }
        for (int l = 0; l < 32; l++) if (wr[l]) slots[(rp[4 * l] >> 20) & 1023] = res[l];
    }
    const uint32_t *op = w.data() + 4 + 2 * nin;
    for (uint32_t e = 0; e < nout; e++) out0[op[2 * e + 1] & 0xffffffu] = slots[op[2 * e]];
}

static void run_program1(const std::vector<uint32_t> &w, const fp *in0, const fp *in1, const fp *cst, fp *out0) {
    const uint32_t nr = w[0], nslots = w[1], nin = w[2], nout = w[3];
    std::vector<fp> slots(nslots);
    fp_set_zero(slots[0]);
    for (uint32_t e = 0; e < nin; e++) {
        uint32_t sl = w[4 + 2 * e], ref = w[5 + 2 * e], buf = ref >> 24, idx = ref & 0xffffffu;
        slots[sl] = (buf == 0 ? in0 : (buf == 1 ? in1 : cst))[idx];
    }
    const uint32_t *rp = w.data() + 4 + 2 * (nin + nout);
    for (uint32_t r = 0; r < nr; r++, rp += 32) {
        fp res[32];
        for (int l = 0; l < 32; l++) {              // all lanes read before any lane writes (stricter than the device)
            uint32_t x = rp[l];
            if (!x) continue;
            if ((x >> 30) == 0) { out0[(((x >> 20) & 1023) << 10) | (x & 1023)] = slots[(x >> 10) & 1023]; continue; }   // STORE
            const fp &a = slots[(x >> 10) & 1023], &b = slots[x & 1023];
            if ((x >> 30) == 1) fp_mul(res[l], a, b); else if ((x >> 30) == 2) fp_add(res[l], a, b); else fp_sub(res[l], a, b);
        }
        for (int l = 0; l < 32; l++) if (rp[l] >> 30) slots[(rp[l] >> 20) & 1023] = res[l];
    }
    const uint32_t *op = w.data() + 4 + 2 * nin;
    for (uint32_t e = 0; e < nout; e++) out0[op[2 * e + 1] & 0xffffffu] = slots[op[2 * e]];
}
static void run_program(const std::vector<uint32_t> &w, const fp *in0, const fp *in1, const fp *cst, fp *out0) {
    if (fpprog::program_format() == 2) run_program2(w, in0, in1, cst, out0); else run_program1(w, in0, in1, cst, out0);
}
// tests run every program in both formats
extern "C" void hs_set_program_format(int f) { fpprog::g_format_override = f; }

static void const_pool(fp *cst) {
    memcpy(cst + fpprog::CONST_FROB1, FROB1, sizeof(FROB1));
    memcpy(cst + fpprog::CONST_FROB2, FROB2, sizeof(FROB2));
    memcpy(cst + fpprog::CONST_FROB3, FROB3, sizeof(FROB3));
    memcpy(cst + fpprog::CONST_PSI_CX, &PSI_CX, sizeof(PSI_CX));
    memcpy(cst + fpprog::CONST_PSI_CY, &PSI_CY, sizeof(PSI_CY));
    memcpy(cst + fpprog::CONST_PSI2_CX, &PSI2_CX, sizeof(PSI2_CX));
    memcpy(cst + fpprog::CONST_ONE, &FP_ONE, sizeof(FP_ONE));
}
// stats[0..3] = rounds, mul rounds, slots, ops
int hs_prog_final(const fp12 *partials, int count, fp12 *out, int *stats) {
    fpprog::Program P = fpprog::build_final(count);
    if (!P.ok) return 0;
    fp cst[fpprog::CONST_COUNT];
    const_pool(cst);
    run_program(P.words, (const fp *)partials, nullptr, cst, (fp *)out);
    stats[0] = P.nrounds; stats[1] = P.nmul_rounds; stats[2] = P.nslots; stats[3] = P.nops;
    return 1;
}
// the device path: norm program -> fp_inv_vartime -> main program reading the inverse from IN1
int hs_prog_final_split(const fp12 *partials, int count, fp12 *out, int *stats) {
    fpprog::Program A = fpprog::build_final(count, fpprog::INV_EMIT_ARG), B = fpprog::build_final(count, fpprog::INV_EXTERNAL);
    if (!A.ok || !B.ok) return 0;
    fp cst[fpprog::CONST_COUNT];
    const_pool(cst);
    fp norm, ninv;
    run_program(A.words, (const fp *)partials, nullptr, cst, &norm);
    fp_inv_vartime(ninv, norm);
    run_program(B.words, (const fp *)partials, &ninv, cst, (fp *)out);
    stats[0] = A.nrounds + B.nrounds; stats[1] = A.nmul_rounds + B.nmul_rounds; stats[2] = B.nslots; stats[3] = A.nops + B.nops;
    return 1;
}
int hs_prog_combine(const fp12 *seg, int nseg, fp12 *out, int *stats) {
    int len[64];
    for (int j = 0; j < nseg; j++) len[j] = ml_seg_hi(j, nseg) - ml_seg_lo(j, nseg) + 1;
    fpprog::Program P = fpprog::build_combine(nseg, len);
    if (!P.ok) return 0;
    fp cst[fpprog::CONST_COUNT];
    const_pool(cst);
    run_program(P.words, (const fp *)seg, nullptr, cst, (fp *)out);
    stats[0] = P.nrounds; stats[1] = P.nmul_rounds; stats[2] = P.nslots; stats[3] = P.nops;
    return 1;
}
// G1 MSM window Horner as a dataflow program: hom = nwin x (X, Y, Z) homogeneous, out = (X, Y, Z) homogeneous
int hs_prog_msm_horner(const fp *hom, int nwin, int c, fp *out5, int *stats) {
    fpprog::Program P = fpprog::build_msm_horner_g1(nwin, c);
    if (!P.ok) return 0;
    run_program(P.words, hom, nullptr, nullptr, out5);
    stats[0] = P.nrounds; stats[1] = P.nmul_rounds; stats[2] = P.nslots; stats[3] = P.nops;
    return 1;
}
// per-set G2 programs of the small-batch route: hom = (X, Y, Z) over Fp2 = 6 fp in, 6 fp out
int hs_prog_g2_clear_cofactor(const fp *hom, fp *out6, int *stats) {
    fpprog::Program P = fpprog::build_g2_clear_cofactor();
    if (!P.ok) return 0;
    fp cst[fpprog::CONST_COUNT];
    const_pool(cst);
    run_program(P.words, hom, nullptr, cst, out6);
    stats[0] = P.nrounds; stats[1] = P.nmul_rounds; stats[2] = P.nslots; stats[3] = P.nops;
    return 1;
}
int hs_prog_g2_mul64(const fp *hom, uint64_t k, fp *out6, int *stats) {
    fpprog::Program P = fpprog::build_g2_mul64();
    if (!P.ok) return 0;
    fp cst[fpprog::CONST_COUNT], bits[64];
    const_pool(cst);
    for (int i = 0; i < 64; i++) { if ((k >> i) & 1) bits[i] = FP_ONE; else fp_set_zero(bits[i]); }
    run_program(P.words, hom, bits, cst, out6);
    stats[0] = P.nrounds; stats[1] = P.nmul_rounds; stats[2] = P.nslots; stats[3] = P.nops;
    return 1;
}
// Miller-loop lines of one pair: the per-pair program against the straight-line miller_lines of pairing.cuh.
// out_prog: 68 x 6 fp; out_ref: 68 x 72 words (stride 1)
int hs_prog_miller_lines(const g2_aff *Q, const g1_aff *P, fp *out_prog, uint32_t *out_ref, int *stats) {
    fpprog::Program Pg = fpprog::build_miller_lines();
    if (!Pg.ok) return 0;
    fp cst[fpprog::CONST_COUNT];
    const_pool(cst);
    run_program(Pg.words, (const fp *)Q, (const fp *)P, cst, out_prog);
    miller_lines(*Q, *P, out_ref, 1);
    stats[0] = Pg.nrounds; stats[1] = Pg.nmul_rounds; stats[2] = Pg.nslots; stats[3] = Pg.nops;
    return 1;
}
int hs_prog_msm_horner_g2(const fp *hom, int nwin, int c, fp *out6, int *stats) {
    fpprog::Program P = fpprog::build_msm_horner_g2(nwin, c);
    if (!P.ok) return 0;
    run_program(P.words, hom, nullptr, nullptr, out6);
    stats[0] = P.nrounds; stats[1] = P.nmul_rounds; stats[2] = P.nslots; stats[3] = P.nops;
    return 1;
}
int hs_prog_fp12_product(const fp12 *in, int count, fp12 *out, int *stats) {
    fpprog::Program P = fpprog::build_fp12_product(count);
    if (!P.ok) return 0;
    run_program(P.words, (const fp *)in, nullptr, nullptr, (fp *)out);
    stats[0] = P.nrounds; stats[1] = P.nmul_rounds; stats[2] = P.nslots; stats[3] = P.nops;
    return 1;
}
int hs_pubkey_from_bytes(const uint8_t *in, int len, int group_check, g1_aff *out) { return pubkey_from_bytes(*out, in, len, group_check != 0); }
int hs_signature_from_bytes(const uint8_t *in, int len, int group_check, g2_aff *out) { return signature_from_bytes(*out, in, len, group_check != 0); }
void hs_g1_compress(const g1_aff *p, uint8_t *out) { g1_compress(out, *p); }
void hs_miller_combine(const fp12 *seg, int nseg, fp12 *out) { miller_combine(*out, seg, nseg); }

// ---- route.hpp: the plans of the batch pipeline and of the MSM and the Miller-loop workspaces, thresholds read from the
// environment at every call ----
// out: the fields of route::batch_plan in declaration order
void hs_plan_batch(size_t n, size_t total_n, uint32_t chunks, int host_src, int scalars, int use_side, int acc_team,
                   int serial_tail, int use_graph, int *out) {
    const route::switches sw = {use_side != 0, acc_team != 0, serial_tail != 0, use_graph != 0};
    const route::batch_plan p = route::plan_batch(route::read_thresholds(), sw, n, total_n, chunks, host_src != 0, scalars != 0);
    const int v[12] = {p.hash, p.sliced, p.small, p.sig, p.g1_aside, p.msm_after_hash, p.defer_sig, p.affine, p.chain_hog,
                       p.chain_wait, p.graph, p.copy_ahead};
    memcpy(out, v, sizeof v);
}
// The routes of every batch of 1 .. n_max sets in a context of as many sets, under the default switches of blsgpu_create
// (side streams, team accumulation, graph replay; no serial tail).  out: n_max rows of 14 ints = the fields of
// route::batch_plan in declaration order, then the lines route of every tile but the last and of the last tile of the
// Miller plan of the pairs the batch runs (n + 1, or n when the signature pair is deferred; blsgpu.cu run_partial_impl).
void hs_plan_routes(size_t n_max, uint32_t chunks, int host_src, int scalars, int *out) {
    const route::thresholds t = route::read_thresholds();
    const route::switches sw = {true, true, false, true};
    for (size_t n = 1; n <= n_max; n++, out += 14) {
        const route::batch_plan p = route::plan_batch(t, sw, n, n, chunks, host_src != 0, scalars != 0);
        const size_t np = p.defer_sig ? n : n + 1;
        const route::miller_plan m = route::plan_miller(t, np, route::miller_caps_batch(t, n).lines_cap, true, false);
        const int v[14] = {p.hash, p.sliced, p.small, p.sig, p.g1_aside, p.msm_after_hash, p.defer_sig, p.affine, p.chain_hog,
                           p.chain_wait, p.graph, p.copy_ahead, m.lines, m.lines_last};
        memcpy(out, v, sizeof v);
    }
}
// 1 if the pair of final-exponentiation programs over `count` partials (norm, then the exponentiation around the
// external inversion) builds within the slot file, as blsgpu.cu run_final_enqueue needs them
int hs_prog_final_builds(int count) {
    return fpprog::build_final(count, fpprog::INV_EMIT_ARG).ok && fpprog::build_final(count, fpprog::INV_EXTERNAL).ok;
}
// out: G, nseg, lines, lines_last, ncols, gt_prog
void hs_plan_miller(size_t np, size_t lines_cap, int team, int serial_tail, long long *out) {
    const route::miller_plan p = route::plan_miller(route::read_thresholds(), np, lines_cap, team != 0, serial_tail != 0);
    const long long v[6] = {p.G, p.nseg, p.lines, p.lines_last, (long long)p.ncols, p.gt_prog};
    memcpy(out, v, sizeof v);
}
// The Miller-loop workspace of a context of max_sets sets (sig == 0) or of the deferred signature pair (sig != 0).
// out: lines_cap, f_cap, f2_cap, small_lines
void hs_miller_caps(size_t max_sets, int sig, long long *out) {
    const route::miller_caps c = sig ? route::miller_caps_sig() : route::miller_caps_batch(route::read_thresholds(), max_sets);
    const long long v[4] = {(long long)c.lines_cap, (long long)c.f_cap, (long long)c.f2_cap, (long long)c.small_lines};
    memcpy(out, v, sizeof v);
}
// the first np in 1 .. np_max whose Miller plan does not fit that workspace, 0 if every plan fits
size_t hs_miller_misfit(size_t max_sets, int sig, size_t np_max, int team, int serial_tail) {
    const route::thresholds t = route::read_thresholds();
    const route::miller_caps c = sig ? route::miller_caps_sig() : route::miller_caps_batch(t, max_sets);
    for (size_t np = 1; np <= np_max; np++)
        if (!route::fits(route::plan_miller(t, np, c.lines_cap, team != 0, serial_tail != 0), c)) return np;
    return 0;
}
// out: c, nwin, B, L, nseg, G, emax, horner_prog, scratch bytes of the G1 and of the G2 MSM, gw0[0..G], K[0..G-1],
// preg[0..G]
void hs_plan_msm(size_t n, int nbits, int sms, long long *out) {
    const route::msm_plan p = route::plan_msm(route::read_thresholds(), n, nbits, sms);
    const long long v[10] = {p.c, p.nwin, (long long)p.B, (long long)p.L, (long long)p.nseg, p.G, (long long)p.emax,
                             p.horner_prog, (long long)route::msm_scratch(p, sizeof(g1_jac)).total,
                             (long long)route::msm_scratch(p, sizeof(g2_jac)).total};
    memcpy(out, v, sizeof v);
    long long *o = out + 10;
    for (int g = 0; g <= p.G; g++) *o++ = p.gw0[g];
    for (int g = 0; g < p.G; g++) *o++ = p.K[g];
    for (int g = 0; g <= p.G; g++) *o++ = (long long)p.preg[g];
}
// The runs of equal MSM shape over n = 1 .. n_max points with nbits-bit scalars on `sms` SMs.  The shape is (c, nwin, L,
// nseg, G, horner_prog, and for every group whether its chunk length K sits at its floor of 8); K above the floor grows
// with n and is not part of it.  out: (first n, last n) of each run, at most cap runs; returns the number of runs, or
// -1 if there are more than cap.
int hs_msm_runs(int nbits, int sms, size_t n_max, long long *out, int cap) {
    const route::thresholds t = route::read_thresholds();
    long long prev[15] = {}, cur[15];
    int runs = 0;
    for (size_t n = 1; n <= n_max; n++) {
        const route::msm_plan p = route::plan_msm(t, n, nbits, sms);
        const long long v[7] = {p.c, p.nwin, (long long)p.L, (long long)p.nseg, p.G, p.horner_prog, 0};
        memcpy(cur, v, sizeof v);
        for (int g = 0; g < 8; g++) cur[7 + g] = g < p.G && p.K[g] == 8;
        if (n == 1 || memcmp(cur, prev, sizeof cur) != 0) {
            if (runs == cap) return -1;
            if (runs) out[2 * runs - 1] = (long long)n - 1;
            out[2 * runs] = (long long)n;
            runs++;
            memcpy(prev, cur, sizeof cur);
        }
    }
    if (runs) out[2 * runs - 1] = (long long)n_max;
    return runs;
}
}
