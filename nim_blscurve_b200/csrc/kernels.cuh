// kernels.cuh — __global__ kernels of the batch-verification pipeline (one signature set per thread).
//
// Stage order (blsgpu.cu launches them on one stream):
//   k_rlc_scalars   A2  blst_min_pubkey_sig_core.nim:476-505,:545-556   one thread per reference chunk
//   k_hash_sets     A3  map_to_g2.c:388-396                               H(m_i), Jacobian
//   k_g1_mul        A5  ec_mult.h:178-223 (G1)                            [r_i] pk_i, Jacobian
//   k_pairs_affine  A4  e2.c:97-112, e1.c:60-75                           one shared inversion per set
//   k_g2_mul        A5  ec_mult.h:178-223 (G2)                            [r_i] sig_i ; k_g2_tree sums them
//   k_sig_pair      A9  aggregate.c:479-495                               (S, -G1) becomes pair number n
//   k_miller_lines  A7  pairing.c:220-261 (line_dbl/line_add/line_by_Px2) 68 line triples per pair, word-major
//   k_miller_acc    A6/A7/A8 pairing.c:253-260, aggregate.c:410-458       per (group, segment) Fp12 + block product
//   k_fp12_rows     A8  GT product per segment row ; k_combine: Horner over segments -> 576-byte rank partial
//   k_final         A9/A10 pairing.c:371-404, fp12_tower.c:773-786        product, final exp, ==1, GT bytes
#pragma once
#include <cuda_runtime.h>
#include "../../include/blsgpu.h"
#include "h2c.cuh"
#include "pairing.cuh"
#include "acc_team.cuh"
#include "io.cuh"
#include "pair_route.cuh"
#include "tma_stage.cuh"
#include "fplin.cuh"

namespace bls {

constexpr int fpprog_const_count = 36;                    // == fpprog::CONST_COUNT (static_assert in blsgpu.cu)

// heavy kernels: at most 128 registers -> 4 blocks of 128 threads (16 warps, 4 per scheduler) per SM
#ifndef BLS_LB_BLOCKS
#define BLS_LB_BLOCKS 4
#endif
#define BLS_LB __launch_bounds__(128, BLS_LB_BLOCKS)

struct sigset { g1_aff pk; uint8_t msg[32]; g2_aff sig; };
static_assert(sizeof(sigset) == 320, "SignatureSet layout (bls_batch_verifier.nim:34)");
static_assert(sizeof(fp12) == 576 && sizeof(g2_jac) == 288 && sizeof(g1_jac) == 144, "layout");

// DST_ETH2 (blscurve/bls_sig_min_pubkey.nim:31): sha256.cuh

struct words8 { uint32_t w[8]; };   // a 32-byte string as big-endian words

// SHA-256 of a 32-byte input held as BE words (one compression)
__device__ __forceinline__ void sha256_of_32(uint32_t *out, const uint32_t *in) {
    uint32_t h[8] = {0x6a09e667u, 0xbb67ae85u, 0x3c6ef372u, 0xa54ff53au, 0x510e527fu, 0x9b05688cu, 0x1f83d9abu, 0x5be0cd19u};
    uint32_t w[16];
#pragma unroll
    for (int i = 0; i < 8; i++) w[i] = in[i];
    w[8] = 0x80000000u;
#pragma unroll
    for (int i = 9; i < 15; i++) w[i] = 0;
    w[15] = 256;
    sha256_block_regs(h, w);
#pragma unroll
    for (int i = 0; i < 8; i++) out[i] = h[i];
}

__device__ __forceinline__ uint64_t le64_of_be_words(const uint32_t *d) {
    // first 8 bytes of the digest read as a little-endian u64
    uint32_t lo = __byte_perm(d[0], 0, 0x0123), hi = __byte_perm(d[1], 0, 0x0123);
    return ((uint64_t)hi << 32) | lo;
}

__device__ __forceinline__ void chunk_range(size_t nchunks, size_t total, size_t cid, size_t &off, size_t &len) {
    size_t base = total / nchunks, rem = total % nchunks;
    if (cid < rem) { off = (base + 1) * cid; len = base + 1; }
    else { off = base * cid + rem; len = base; }
}

// One thread per reference chunk walks that chunk's sequential SHA-256 chain and stores the scalars of
// the indices this rank owns ([first, first+n) of the global batch).
// d_srb (nullable): the 32 random bytes as 8 big-endian words in device memory instead of the by-value copy — the
// form a captured CUDA graph needs, where kernel arguments are frozen but the bytes change with every call.
// started (nullable): set to 1 by the first thread as soon as the block runs (k_wait_started on the main stream holds the
// hash kernel back until then, so that the block of chains gets its SM before the machine is full).
__device__ __forceinline__ unsigned long long gtimer() { unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); return t; }
__device__ __forceinline__ unsigned smid() { unsigned v; asm volatile("mov.u32 %0, %%smid;" : "=r"(v)); return v; }
__device__ __forceinline__ void rlc_chains(words8 &srb, const uint32_t *d_srb, size_t total_n, uint32_t chunks, size_t first,
                                           size_t n, uint64_t *out, unsigned long long *dbg, size_t block) {
    if (d_srb) for (int k = 0; k < 8; k++) srb.w[k] = d_srb[k];
    size_t nb = chunks == 0 ? 1 : (total_n < chunks ? total_n : (size_t)chunks);
    size_t c = block * blockDim.x + threadIdx.x;
    if (c >= nb) return;
    size_t off, len;
    chunk_range(nb, total_n, c, off, len);
    if (off >= first + n || off + len <= first) return;
    uint32_t seed[8];
    if (chunks == 0) {
        sha256_of_32(seed, srb.w);
    } else {                                           // SHA256(srb || LE64(c)): 40 bytes, one block
        uint32_t h[8] = {0x6a09e667u, 0xbb67ae85u, 0x3c6ef372u, 0xa54ff53au, 0x510e527fu, 0x9b05688cu, 0x1f83d9abu, 0x5be0cd19u};
        uint32_t w[16];
        for (int i = 0; i < 8; i++) w[i] = srb.w[i];
        w[8] = __byte_perm((uint32_t)c, 0, 0x0123);
        w[9] = __byte_perm((uint32_t)((uint64_t)c >> 32), 0, 0x0123);
        w[10] = 0x80000000u;
        for (int i = 11; i < 15; i++) w[i] = 0;
        w[15] = 320;
        sha256_block(h, w);
        for (int i = 0; i < 8; i++) seed[i] = h[i];
    }
    for (size_t i = off; i < off + len; i++) {
        uint64_t r;
        do {
            uint32_t t[8];
            sha256_of_32(t, seed);
#pragma unroll
            for (int k = 0; k < 8; k++) seed[k] = t[k];
            r = le64_of_be_words(seed);
        } while (r == 0);
        if (i >= first && i < first + n) out[i - first] = r;
    }
    if (dbg && c == 0) dbg[1] = gtimer();
}
// started (nullable): set to 1 by the first thread as soon as the block runs (k_wait_started on the main stream holds the
// hash kernel back until then, so that the block of chains gets its SM before the machine is full).
// dbg (nullable, BLSGPU_DEBUG_CHAIN): %globaltimer at start and end, SM number.
// Measured with it (round 2): the lone chain warp is slowed by the code the OTHER SM of its TPC runs — 12.8 ms alone,
// 13.9 / 23.1 ms beside two builds of the hash kernel that differ only in code size, 13.3 ms with the partner SM held
// idle (by a 2-block cluster or by a guard block): the 21 KB unrolled SHA-256 loop lives in an instruction cache level
// the two SMs of a TPC share.  Holding the partner idle is NOT adopted: with a whole TPC out of the machine the
// two-wave hash kernel takes 26.9-28.4 ms instead of 24.0 (one SM out: 24.0), more than the chain gains.
__global__ void k_rlc_scalars(words8 srb, const uint32_t *d_srb, size_t total_n, uint32_t chunks, size_t first, size_t n,
                              uint64_t *out, volatile int *started, unsigned long long *dbg = nullptr) {
    if (started && blockIdx.x == 0 && threadIdx.x == 0) { *started = 1; __threadfence(); }
    if (dbg && blockIdx.x == 0 && threadIdx.x == 0) { dbg[0] = gtimer(); dbg[3] = smid(); }
    rlc_chains(srb, d_srb, total_n, chunks, first, n, out, dbg, blockIdx.x);
}

// One thread polls the flag the chain kernel raises when its block is resident; gives up after `budget` clock cycles
// (the chain may be queued behind other work on a busy device: then the hash simply goes first, as without this).
__global__ void k_wait_started(volatile int *started, long long budget, unsigned long long *dbg = nullptr) {
    if (blockIdx.x != 0 || threadIdx.x != 0) return;
    const long long t0 = clock64();
    while (*started == 0 && clock64() - t0 < budget) __nanosleep(200);
    if (dbg) { dbg[2] = gtimer(); dbg[4] = *started; }
}

// Blinding scalars of MultiSignatureSet.combine (blst_min_pubkey_sig_core.nim:590-606): seed <- SHA256(seed), the
// digest is read as four little-endian u64 and consumed from the LAST one down; zeros are skipped.  Sequential chain.
__global__ void k_combine_scalars(words8 srb, size_t n, uint64_t *out) {
    if (blockIdx.x != 0 || threadIdx.x != 0) return;
    uint32_t seed[8];
    for (int k = 0; k < 8; k++) seed[k] = srb.w[k];
    int avail = 0;
    for (size_t i = 0; i < n; i++) {
        for (;;) {
            if (avail == 0) {
                uint32_t t[8];
                sha256_of_32(t, seed);
                for (int k = 0; k < 8; k++) seed[k] = t[k];
                avail = 4;
            }
            avail--;
            uint64_t v = le64_of_be_words(seed + 2 * avail);
            if (v != 0) { out[i] = v; break; }
        }
    }
}

// The 128 messages of the block (32 of the 320 bytes of each record) are staged into shared memory by TMA bulk copies
// (tma_stage.cuh), 4 KB per block.
__global__ void BLS_LB k_hash_sets(const sigset *sets, size_t n, g2_jac *H) {
    __shared__ __align__(128) uint8_t tile[128 * 32];
    __shared__ uint64_t bar;
    const size_t base = (size_t)blockIdx.x * blockDim.x;
    const size_t cnt = n - base < blockDim.x ? n - base : blockDim.x;
    tma_stage_rows(tile, 32, sets[base].msg, sizeof(sigset), (uint32_t)cnt, &bar);
    size_t i = base + threadIdx.x;
    if (i >= n) return;
    alignas(16) uint8_t msg[32];
    {
        const uint4 *m = (const uint4 *)(tile + 32 * threadIdx.x);
        uint4 m0 = m[0], m1 = m[1];
        *(uint4 *)msg = m0;
        *(uint4 *)(msg + 16) = m1;
    }
    g2_jac h;
    hash_to_g2_jac_eth2(h, msg);
    H[i] = h;
}

// Small batches: two lanes per message, one SSWU map each (the two maps of hash_to_curve are independent and are a
// fifth of the serial work); the odd lane hands its point to the even lane, which adds, applies the isogeny and clears
// the cofactor.  Same result as k_hash_sets; used while 2n threads still leave the machine under-filled.
__global__ void BLS_LB k_hash_sets_pair(const sigset *sets, size_t n, g2_jac *H) {
    const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t i = t >> 1;
    const bool odd = t & 1;
    const bool live = i < n;
    uint8_t msg[32], dst[43];
    for (int k = 0; k < 32; k++) msg[k] = live ? sets[i].msg[k] : 0;
    for (int k = 0; k < 43; k++) dst[k] = DST_ETH2[k];
    fp2 u0, u1;
    hash_to_field_fp2x2(u0, u1, msg, 32, dst, 43);
    g2_jac q, other;
    sswu_g2(q, odd ? u1 : u0);
    {
        uint32_t *d = (uint32_t *)&other;
        const uint32_t *sp = (const uint32_t *)&q;
        for (int k = 0; k < (int)(sizeof(g2_jac) / 4); k++) d[k] = __shfl_down_sync(0xffffffffu, sp[k], 1);
    }
    if (odd || !live) return;
    pt_add(q, q, other, &SSWU_A);
    iso3_g2(q, q);
    g2_jac h;
    g2_clear_cofactor(h, q);
    H[i] = h;
}

// ---- mid-size route: two lanes per set (fp2h.cuh / pair_route.cuh) --------------------------------------------------
// H(m_i) with every Fp2 operation split over a lane pair; lane pair t/2 owns set t/2.  Output identical to k_hash_sets.
__global__ void BLS_LB k_hash_sets_lanes2(const sigset *sets, size_t n, g2_jac *H) {
    __shared__ __align__(128) uint8_t tile[64 * 32];       // the block's 64 messages, TMA bulk copies (tma_stage.cuh)
    __shared__ uint64_t bar;
    const size_t base = (size_t)blockIdx.x * (blockDim.x >> 1);
    const size_t cnt = n - base < (blockDim.x >> 1) ? n - base : (blockDim.x >> 1);
    tma_stage_rows(tile, 32, sets[base].msg, sizeof(sigset), (uint32_t)cnt, &bar);
    const size_t i = base + (threadIdx.x >> 1);
    if (i >= n) return;                                    // both lanes of a pair leave together
    alignas(16) uint8_t msg[32];
    {
        const uint4 *m = (const uint4 *)(tile + 32 * (threadIdx.x >> 1));
        *(uint4 *)msg = m[0];
        *(uint4 *)(msg + 16) = m[1];
    }
    g2h_jac h;
    hash_to_g2_pair(h, msg, 32, nullptr, 0);
    fp *out = (fp *)&H[i] + (h_odd() ? 1 : 0);             // g2_jac = x.c0 x.c1 y.c0 y.c1 z.c0 z.c1
    out[0] = h.x.v;
    out[2] = h.y.v;
    out[4] = h.z.v;
}
// the 68 line triples of pair t/2, word for word those of k_miller_lines
__global__ void __launch_bounds__(128, BLS_LB_BLOCKS) k_miller_lines_lanes2(const g2_aff *Q, const g1_aff *P, size_t np,
                                                                            uint32_t *lines, size_t stride) {
    const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t p = t >> 1;
    if (p >= np) return;
    const fp *q = (const fp *)&Q[p] + (h_odd() ? 1 : 0);   // g2_aff = x.c0 x.c1 y.c0 y.c1
    g2h_aff qh;
    qh.x.v = q[0];
    qh.y.v = q[2];
    g1_aff a = P[p];
    const bool inf = (f_is_zero(qh.x) & f_is_zero(qh.y)) | aff_is_inf(a);
    miller_lines_pair(qh, a, inf, lines + p, stride);
}

// ---- small-batch route (<= 1024 sets): the long serial stretches run as per-set dataflow programs ----
// homogeneous (X : Y : Z) over Fp2 <- Jacobian; infinity -> (0 : 1 : 0)
BLS_NOINLINE void g2_jac_to_hom(fp *hom, const g2_jac &p) {
    fp2 x, y, z;
    if (pt_is_inf(p)) {
        fp2_set_zero(x); fp2_set_zero(y); y.c0 = FP_ONE; fp2_set_zero(z);
    } else {
        fp2 z2;
        fp2_mul(x, p.x, p.z);
        y = p.y;
        fp2_sqr(z2, p.z);
        fp2_mul(z, z2, p.z);
    }
    hom[0] = x.c0; hom[1] = x.c1; hom[2] = y.c0; hom[3] = y.c1; hom[4] = z.c0; hom[5] = z.c1;
}
// first half of k_hash_sets_pair: XMD, one SSWU map per lane, sum on E2', 3-isogeny; the cofactor clearing follows
// as a program (fpprog.hpp build_g2_clear_cofactor)
__global__ void BLS_LB k_hash_map_pair(const sigset *sets, size_t n, fp *hom) {
    const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t i = t >> 1;
    const bool odd = t & 1;
    const bool live = i < n;
    uint8_t msg[32], dst[43];
    for (int k = 0; k < 32; k++) msg[k] = live ? sets[i].msg[k] : 0;
    for (int k = 0; k < 43; k++) dst[k] = DST_ETH2[k];
    fp2 u0, u1;
    hash_to_field_fp2x2(u0, u1, msg, 32, dst, 43);
    g2_jac q, other;
    sswu_g2(q, odd ? u1 : u0);
    {
        uint32_t *d = (uint32_t *)&other;
        const uint32_t *sp = (const uint32_t *)&q;
        for (int k = 0; k < (int)(sizeof(g2_jac) / 4); k++) d[k] = __shfl_down_sync(0xffffffffu, sp[k], 1);
    }
    if (odd || !live) return;
    pt_add(q, q, other, &SSWU_A);
    iso3_g2(q, q);
    g2_jac_to_hom(hom + 6 * i, q);
}
// The same on lane pairs with every Fp2 operation split over the two lanes (pair_route.cuh): the two square-root chains
// still run one map per lane, and the Fp2 stretches around them (SSWU, sum on E2', isogeny) take half as long.
// msgs == nullptr: the messages are those of the signature sets (32 bytes, DST of bls_sig_min_pubkey.nim:31).
__global__ void BLS_LB k_hash_map_lanes2(const sigset *sets, const uint8_t *msgs, const uint32_t *offs, const uint8_t *dst_g,
                                         uint32_t dst_len, size_t n, fp *hom) {
    const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t i = t >> 1;
    if (i >= n) return;
    g2h_jac q;
    if (msgs) {
        hash_map_to_e2_pair(q, msgs + offs[i], offs[i + 1] - offs[i], dst_g, dst_len);
    } else {
        uint8_t msg[32];
        for (int k = 0; k < 32; k++) msg[k] = sets[i].msg[k];
        hash_map_to_e2_pair(q, msg, 32, nullptr, 0);
    }
    fp2h X, Y, Z;
    jac_to_hom_pair(X, Y, Z, q);
    fp *out = hom + 6 * i + (h_odd() ? 1 : 0);
    out[0] = X.v;
    out[2] = Y.v;
    out[4] = Z.v;
}
// the same for the verify entry points: arbitrary messages (msgs + offs[i] .. offs[i+1]) and domain separation tag
__global__ void BLS_LB k_hash_map_pair_msgs(const uint8_t *msgs, const uint32_t *offs, const uint8_t *dst, uint32_t dst_len,
                                            size_t n, fp *hom) {
    const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t i = t >> 1;
    const bool odd = t & 1;
    const bool live = i < n;
    const size_t j = live ? i : 0;
    fp2 u0, u1;
    hash_to_field_fp2x2(u0, u1, msgs + offs[j], offs[j + 1] - offs[j], dst, dst_len);
    g2_jac q, other;
    sswu_g2(q, odd ? u1 : u0);
    {
        uint32_t *d = (uint32_t *)&other;
        const uint32_t *sp = (const uint32_t *)&q;
        for (int k = 0; k < (int)(sizeof(g2_jac) / 4); k++) d[k] = __shfl_down_sync(0xffffffffu, sp[k], 1);
    }
    if (odd || !live) return;
    pt_add(q, q, other, &SSWU_A);
    iso3_g2(q, q);
    g2_jac_to_hom(hom + 6 * i, q);
}
// homogeneous (X : Y : Z) -> affine (X / Z, Y / Z), one working lane per warp-sized block (binary-Euclid inversion)
__global__ void k_g2_hom_to_affine(const fp *hom, size_t n, g2_aff *out) {
    if (threadIdx.x != 0 || blockIdx.x >= n) return;
    const fp *h = hom + 6 * (size_t)blockIdx.x;
    fp2 X, Y, Z, zi;
    X.c0 = h[0]; X.c1 = h[1]; Y.c0 = h[2]; Y.c1 = h[3]; Z.c0 = h[4]; Z.c1 = h[5];
    g2_aff a;
    fp2_inv_vartime(zi, Z);                 // Z = 0 -> 0 -> the all-zero affine encoding of infinity
    fp2_mul(a.x, X, zi);
    fp2_mul(a.y, Y, zi);
    out[blockIdx.x] = a;
}
// homogeneous (X : Y : Z) -> Jacobian (X Z, Y Z^2, Z); Z = 0 -> infinity
__global__ void k_g2_hom_to_jac(const fp *hom, size_t n, g2_jac *out) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const fp *h = hom + 6 * i;
    fp2 X, Y, Z;
    X.c0 = h[0]; X.c1 = h[1]; Y.c0 = h[2]; Y.c1 = h[3]; Z.c0 = h[4]; Z.c1 = h[5];
    g2_jac j;
    if (fp2_is_zero(Z)) pt_set_inf(j);
    else { fp2 z2; fp2_mul(j.x, X, Z); fp2_sqr(z2, Z); fp2_mul(j.y, Y, z2); j.z = Z; }
    out[i] = j;
}
// inputs of the [r_i] sig_i program (build_g2_mul64): the signature as (x : y : 1) (infinity (0 : 1 : 0)) and the 64
// scalar bits as field elements 0 / 1
__global__ void k_g2_mul_prep(const sigset *sets, const uint64_t *r, size_t n, fp *hom, fp *bits) {
    const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t i = t >> 6;
    const int b = (int)(t & 63);
    if (i >= n) return;
    fp v;
    if ((r[i] >> b) & 1) v = FP_ONE; else fp_set_zero(v);
    bits[64 * i + b] = v;
    if (b == 0) {
        g2_aff a = sets[i].sig;
        g2_jac j;
        pt_from_affine(j, a);
        g2_jac_to_hom(hom + 6 * i, j);
    }
}

__global__ void BLS_LB k_g1_mul(const sigset *sets, const uint64_t *r, size_t n, g1_jac *Pj, int *flags) {
    __shared__ __align__(128) sigset tile[128];            // the block's 128 sets, one TMA bulk copy (tma_stage.cuh)
    __shared__ uint64_t bar;
    const size_t base = (size_t)blockIdx.x * blockDim.x;
    const size_t cnt = n - base < blockDim.x ? n - base : blockDim.x;
    tma_stage_tile(tile, sets + base, (uint32_t)(cnt * sizeof(sigset)), &bar);
    size_t i = base + threadIdx.x;
    if (i >= n) return;
    g1_aff pk = tile[threadIdx.x].pk;
    if (aff_is_inf(pk)) atomicOr(flags, 1);            // BLST_PK_IS_INFINITY (aggregate.c:296)
    g1_jac j;
    pt_mul_u64_w4(j, pk, r[i]);
    Pj[i] = j;
}

// H_i and [r_i]pk_i to affine.  Montgomery's trick twice over: per set the two denominators N(Z_H) and Z_P share
// one inverse, and every thread walks AFF_B sets (strided by the thread count, so that warps stay coalesced) and
// shares ONE Fermat inversion among them: 1 inversion + ~45 multiplications per set become 1/8 inversion + ~50.
#define AFF_B 8
// `spread` (small batches): one working lane per warp-sized block, so that the branchy binary-Euclid inversion of
// different sets never shares a warp (0.15 ms instead of the 0.46 ms of one Fermat chain).
// `per` <= AFF_B sets per thread.  vartime == 2 ("block" mode, batches past the small route): Montgomery's trick a THIRD
// time, across the 128 threads of a block — inclusive prefix and suffix products of the threads' totals through shared
// memory (seven doubling steps), ONE binary-Euclid inversion by thread 0 (0.1 ms, no divergence: one lane works), and
// 1 / total_t = 1 / block_total * prefix_(t-1) * suffix_(t+1).  The 444-step Fermat chain per thread (0.46 ms of pure
// latency whatever the batch size) becomes ~0.12 ms per block.
__global__ void BLS_LB k_pairs_affine(const g2_jac *H, const g1_jac *Pj, size_t n, g2_aff *Q, g1_aff *P, int vartime, int spread,
                                      int per) {
    __shared__ fp sc[2][128];
    __shared__ fp sinv;
    size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x, nthreads = (size_t)gridDim.x * blockDim.x;
    if (spread) {
        if (threadIdx.x != 0) return;
        t = blockIdx.x;
        nthreads = gridDim.x;
    }
    const bool block_mode = vartime == 2;
    if (t >= n && !block_mode) return;
    fp nz[AFF_B], zp[AFF_B], pre[AFF_B];
    int cnt = 0;
    for (int k = 0; k < per; k++) {
        const size_t i = t + (size_t)k * nthreads;
        if (i >= n) break;
        fp2 hz = H[i].z;
        fp a, b;
        fp_sqr_ni(a, hz.c0);
        fp_sqr_ni(b, hz.c1);
        fp_add(a, a, b);                                    // N(Z_H)
        b = Pj[i].z;
        if (fp_is_zero(a)) a = FP_ONE;                      // infinity: keep the product invertible
        if (fp_is_zero(b)) b = FP_ONE;
        nz[k] = a;
        zp[k] = b;
        fp c;
        fp_mul_ni(c, a, b);
        if (k) fp_mul_ni(pre[k], pre[k - 1], c); else pre[k] = c;
        cnt = k + 1;
    }
    fp inv;
    if (block_mode) {
        const int tid = threadIdx.x;
        fp tot;
        if (cnt) tot = pre[cnt - 1]; else tot = FP_ONE;
        sc[0][tid] = tot;
        sc[1][tid] = tot;
        __syncthreads();
        for (int d = 1; d < 128; d <<= 1) {
            fp a, b, x, y;
            const bool ha = tid >= d, hb = tid + d < 128;
            if (ha) { a = sc[0][tid - d]; x = sc[0][tid]; }
            if (hb) { b = sc[1][tid + d]; y = sc[1][tid]; }
            __syncthreads();
            if (ha) { fp_mul_ni(x, x, a); sc[0][tid] = x; }
            if (hb) { fp_mul_ni(y, y, b); sc[1][tid] = y; }
            __syncthreads();
        }
        if (tid == 0) { fp all = sc[0][127], r; fp_inv_vartime(r, all); sinv = r; }
        __syncthreads();
        inv = sinv;
        if (tid > 0) { fp a = sc[0][tid - 1]; fp_mul_ni(inv, inv, a); }
        if (tid < 127) { fp b = sc[1][tid + 1]; fp_mul_ni(inv, inv, b); }
        if (!cnt) return;
    } else if (vartime) fp_inv_vartime(inv, pre[cnt - 1]);
    else fp_inv(inv, pre[cnt - 1]);
    for (int k = cnt - 1; k >= 0; k--) {
        const size_t i = t + (size_t)k * nthreads;
        fp ik, ninv, zpinv, tt;
        if (k) {
            fp_mul_ni(ik, inv, pre[k - 1]);                 // 1 / (N(Z_H) Z_P) of set k
            fp_mul_ni(tt, nz[k], zp[k]);
            fp_mul_ni(inv, inv, tt);
        } else {
            ik = inv;
        }
        fp_mul_ni(ninv, ik, zp[k]);                         // 1/N(Z_H)
        fp_mul_ni(zpinv, ik, nz[k]);                        // 1/Z_P
        g2_jac h = H[i];
        g1_jac p = Pj[i];
        fp2 zhinv;
        fp_mul_ni(zhinv.c0, h.z.c0, ninv);
        fp_mul_ni(tt, h.z.c1, ninv);
        fp_neg(zhinv.c1, tt);
        g2_aff q;
        g1_aff a;
        pt_to_affine_zinv(q, h, zhinv);                     // infinity (Z = 0) -> all-zero affine
        pt_to_affine_zinv(a, p, zpinv);
        Q[i] = q;
        P[i] = a;
    }
}

__global__ void BLS_LB k_g2_mul(const sigset *sets, const uint64_t *r, size_t n, g2_jac *S) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    g2_aff sig = sets[i].sig;
    g2_jac j;
    pt_mul_u64(j, sig, r[i]);                           // infinite signature contributes nothing (aggregate.c:261)
    S[i] = j;
}

// pairwise tree step: x[i] (op)= x[i + half] for i + half < n
__global__ void BLS_LB k_g2_tree(g2_jac *S, size_t n, size_t half) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= half || i + half >= n) return;
    g2_jac a = S[i], b = S[i + half];
    pt_add(a, a, b);
    S[i] = a;
}

__global__ void BLS_LB k_g1_tree(g1_jac *S, size_t n, size_t half) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= half || i + half >= n) return;
    g1_jac a = S[i], b = S[i + half];
    pt_add(a, a, b);
    S[i] = a;
}

__global__ void BLS_LB k_fp12_tree(fp12 *F, size_t n, size_t half) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= half || i + half >= n) return;
    fp12 a = F[i], b = F[i + half];
    fp12_mul(a, a, b);
    F[i] = a;
}

// ---- split Miller loop (pairing.cuh): lines per pair, then accumulation per (group, segment) ----

// The signature-side pair of aggregate.c:479-495, folded into the multi-Miller product as pair number n:
// Q[n] = S (affine), P[n] = -G1.  FE(ML(S,-G1)) = FE(conj(ML(S,G1))), so the post-FE GT is unchanged.
__global__ void k_sig_pair(const g2_jac *S, size_t n, g2_aff *Q, g1_aff *P) {
    if (blockIdx.x != 0 || threadIdx.x != 0) return;
    g2_jac s = *S;
    g2_aff sa;
    pt_to_affine_vt(sa, s);                              // S = infinity -> all-zero -> neutral lines
    Q[n] = sa;
    g1_aff g;
    g.x = G1_GEN_X;
    fp_neg(g.y, G1_GEN_Y);
    P[n] = g;
}

#ifndef BLS_LINES_BLOCKS
#define BLS_LINES_BLOCKS 4
#endif
__global__ void __launch_bounds__(128, BLS_LINES_BLOCKS) k_miller_lines(const g2_aff *Q, const g1_aff *P, size_t np,
                                                                       uint32_t *lines, size_t stride) {
    size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= np) return;
    g2_aff q = Q[p];
    g1_aff a = P[p];
    miller_lines(q, a, lines + p, stride);
}

// Small-batch route: the lines come out of the per-pair program (fpprog.hpp build_miller_lines) as 68 x 6 field
// elements per pair; scatter them into the word-major layout the accumulation reads, substituting the neutral line
// (1, 0, 0) for pairs with a point at infinity (pairing.c:233-241), which the branch-free program cannot express.
__global__ void k_lines_from_prog(const uint32_t *prog_out, const g2_aff *Q, const g1_aff *P, size_t np, uint32_t *lines,
                                  size_t stride) {
    const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t per = (size_t)ML_NLINES * ML_LINE_WORDS;
    if (t >= np * per) return;
    const size_t p = t % np, sw = t / np;
    uint32_t v;
    if (aff_is_inf(Q[p]) | aff_is_inf(P[p])) {
        const int w = (int)(sw % ML_LINE_WORDS);
        v = w < 12 ? FP_ONE.l[w] : 0u;
    } else {
        v = prog_out[p * per + sw];
    }
    lines[sw * stride + p] = v;
}

#define BLS_ACC_BS 128
#ifndef BLS_ACC_BLOCKS
#define BLS_ACC_BLOCKS 2
#endif
// product of the block's Fp12 values through shared memory (word-major, conflict-free); result in thread 0
// `live` = number of threads holding a value other than one (they are the lowest thread indices): the tree starts at
// the smallest power of two that covers them, so a batch of a few pairs does not pay seven levels of products by one
__device__ __forceinline__ void block_fp12_product(fp12 &f, uint32_t *sm, int live = BLS_ACC_BS) {
    const int tid = threadIdx.x;
    int top = BLS_ACC_BS / 2;
    while (top >= 1 && top >= live) top >>= 1;
    for (int half = top; half >= 1; half >>= 1) {
        if (tid >= half && tid < 2 * half) {
            const uint32_t *w = (const uint32_t *)&f;
            for (int k = 0; k < 144; k++) sm[k * half + (tid - half)] = w[k];
        }
        __syncthreads();
        if (tid < half) {
            fp12 b;
            uint32_t *w = (uint32_t *)&b;
            for (int k = 0; k < 144; k++) w[k] = sm[k * half + tid];
            fp12_mul(f, f, b);
        }
        __syncthreads();
    }
}

// grid = (ceil(ngroups / 128), nseg).  Thread (g, j) folds the lines of group g over segment j, the block multiplies
// its 128 values and writes one Fp12 to Fseg[j * row_stride + col_off + blockIdx.x].
__global__ void __launch_bounds__(BLS_ACC_BS, BLS_ACC_BLOCKS) k_miller_acc(const uint32_t *lines, size_t stride, size_t np,
                                                                           size_t ngroups, int G, int nseg, fp12 *Fseg,
                                                                           size_t row_stride, size_t col_off) {
    __shared__ uint32_t sm[(BLS_ACC_BS / 2) * 144];
    const size_t g = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int j = blockIdx.y;
    fp12 f;
    if (g < ngroups) miller_accumulate(f, lines, stride, np, g, ngroups, G, ml_seg_hi(j, nseg), ml_seg_lo(j, nseg));
    else fp12_set_one(f);
    block_fp12_product(f, sm);
    if (threadIdx.x == 0) Fseg[(size_t)j * row_stride + col_off + blockIdx.x] = f;
}

// Team version of the accumulation (acc_team.cuh): grid = (ceil(ngroups / ACC_TPB), nseg); every team of six lanes folds
// the lines of ONE group over ONE segment and writes its Fp12 to Fteam[j * row_stride + col_off + team].
#ifndef BLS_ACCT_BLOCKS
#define BLS_ACCT_BLOCKS 3
#endif
__global__ void __launch_bounds__(ACC_BS, BLS_ACCT_BLOCKS) k_miller_acc_team(const uint32_t *lines, size_t stride, size_t np,
                                                                            size_t ngroups, int G, int nseg, fp12 *Fteam,
                                                                            size_t row_stride, size_t col_off) {
    __shared__ acc_team_sm sm[ACC_TPB];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (lane >= 6 * ACC_TPW) return;                       // lanes 30, 31 idle (never reach a barrier)
    const uint32_t mask = (1u << (6 * ACC_TPW)) - 1;
    const int team = lane / 6, k = lane % 6;
    acc_team_sm &T = sm[warp * ACC_TPW + team];
    const size_t g = ((size_t)blockIdx.x * (ACC_BS / 32) + warp) * ACC_TPW + team;
    const int j = blockIdx.y, i_hi = ml_seg_hi(j, nseg), i_lo = ml_seg_lo(j, nseg);
    const bool team_valid = g < ngroups;
    bool first = true;
    for (int i = i_hi; i >= i_lo; i--) {
        if (!first) team_square(T, k, mask);
        const int s0 = ml_line_index(i), nl = 1 + ml_bit(i);
        for (int a = 0; a < nl; a++)
            for (int kk = 0; kk < G; kk++) {
                // stage the line: lane k fetches Fp number k of the triple (neutral line 1 when the pair does not exist)
                const size_t p = g + (size_t)kk * ngroups;
                fp v;
                if (team_valid && p < np) {
                    const uint32_t *src = lines + ((size_t)(s0 + a) * ML_LINE_WORDS + 12 * k) * stride + p;
#pragma unroll
                    for (int w = 0; w < 12; w++) v.l[w] = src[(size_t)w * stride];
                } else if (k == 0) {
                    v = FP_ONE;
                } else {
                    fp_set_zero(v);
                }
                T.l[k] = v;
                __syncwarp(mask);
                if (k < 3) { fp sum; fp_add(sum, T.l[2 * k], T.l[2 * k + 1]); T.l[6 + k] = sum; }
                __syncwarp(mask);
                if (first) {                                // f = line: w^0 <- l0, w^2 <- l1, w^3 <- l2
                    fp c0, c1;
                    const int li = k == 0 ? 0 : (k == 2 ? 1 : (k == 3 ? 2 : -1));
                    if (li >= 0) { c0 = T.l[2 * li]; c1 = T.l[2 * li + 1]; } else { fp_set_zero(c0); fp_set_zero(c1); }
                    team_store_coeff(T, k, c0, c1);
                    __syncwarp(mask);
                    first = false;
                } else {
                    team_mul_line(T, k, mask);
                }
            }
    }
    if (team_valid) {                                       // coefficient of w^k is a[k&1][k>>1] of the tower layout
        fp2 *dst = (fp2 *)&Fteam[(size_t)j * row_stride + col_off + g];
        fp2 out;
        out.c0 = T.f[k][FV_C0];
        out.c1 = T.f[k][FV_C1];
        dst[3 * (k & 1) + (k >> 1)] = out;
    }
}

// pairwise block reduction of rows: grid = (ceil(ncols / 128), nrows); block b of row j multiplies entries
// [128 b, 128 b + 128) of the row and writes the product to out[j * out_stride + b]
__global__ void __launch_bounds__(BLS_ACC_BS, BLS_ACC_BLOCKS) k_fp12_rows_step(const fp12 *in, size_t in_stride, size_t ncols,
                                                                               fp12 *out, size_t out_stride) {
    __shared__ uint32_t sm[(BLS_ACC_BS / 2) * 144];
    const size_t c = (size_t)blockIdx.x * BLS_ACC_BS + threadIdx.x;
    fp12 f;
    if (c < ncols) f = in[(size_t)blockIdx.y * in_stride + c]; else fp12_set_one(f);
    block_fp12_product(f, sm);
    if (threadIdx.x == 0) out[(size_t)blockIdx.y * out_stride + blockIdx.x] = f;
}

// rows of F padded to `stride` columns: columns [ncols, stride) of row blockIdx.x become one (small-batch GT product)
__global__ void k_fp12_pad_one(fp12 *F, size_t stride, size_t ncols) {
    const size_t c = ncols + threadIdx.x;
    if (c >= stride) return;
    fp12 one;
    fp12_set_one(one);
    F[(size_t)blockIdx.x * stride + c] = one;
}

// one block per segment row: product of ncols values -> seg[j]
__global__ void __launch_bounds__(BLS_ACC_BS, BLS_ACC_BLOCKS) k_fp12_rows(const fp12 *Fseg, size_t row_stride, size_t ncols,
                                                                          fp12 *seg) {
    __shared__ uint32_t sm[(BLS_ACC_BS / 2) * 144];
    const fp12 *row = Fseg + (size_t)blockIdx.x * row_stride;
    fp12 f;
    fp12_set_one(f);
    bool have = false;
    for (size_t c = threadIdx.x; c < ncols; c += BLS_ACC_BS) {
        fp12 b = row[c];
        if (have) fp12_mul(f, f, b); else { f = b; have = true; }
    }
    block_fp12_product(f, sm, ncols < BLS_ACC_BS ? (int)ncols : BLS_ACC_BS);
    if (threadIdx.x == 0) seg[blockIdx.x] = f;
}

// rank partial = conj(prod_j seg[j]^(2^lo_j))   (single thread; 63 Fp12 squarings)
__global__ void k_combine(const fp12 *seg, int nseg, fp12 *out) {
    if (blockIdx.x != 0 || threadIdx.x != 0) return;
    fp12 F;
    miller_combine(F, seg, nseg);
    *out = F;
}

// neutral partial for an empty share: GT one in the in-memory (Montgomery) layout
__global__ void k_partial_one(fp12 *out, int *flag_out) {
    if (blockIdx.x != 0 || threadIdx.x != 0) return;
    fp12 one;
    fp12_set_one(one);
    *out = one;
    if (flag_out) *flag_out = 0;
}
// Seal a rank partial: a share that saw an infinite public key (flag set, aggregate.c:296) emits the ZERO element of
// Fp12 instead of its Miller value.  Zero absorbs the product of the gathered partials and the final exponentiation maps
// it to zero, which is not one: the batch is rejected with an all-zero GT by whoever finalises, so the 576-byte partial
// is the only thing ranks have to exchange (one collective).  The flag is still copied out for callers that want it.
__global__ void k_partial_seal(const int *flags, uint32_t *partial, int *flag_out) {
    const int f = flags[0];
    if (flag_out && threadIdx.x == 0) *flag_out = f;
    if (f) for (int w = threadIdx.x; w < 144; w += blockDim.x) partial[w] = 0u;
}

// ---- warp-cooperative tail: interpreter for the Fp dataflow programs compiled by fpprog.hpp ----
// One warp; field elements live in 48-byte shared-memory slots (slot 0 = zero).  Every round holds at most 32
// independent operations of one kind (32 words per round, word = op:2 | dst:10 | a:10 | b:10, 0 = idle); lane l executes
// operation l.  A slot written
// in round r is never read in round r (fpprog.hpp frees slots only after their last reading round), so one warp
// barrier per round orders everything.
// constant table of the dataflow programs (fpprog::CONST_*), copied from the __constant__ tables of consts.cuh
__global__ void k_fill_consts(fp *dst) {
    const int t = threadIdx.x;
    if (t >= fpprog_const_count) return;
    const fp *src;
    int k;
    if (t < 10) { src = (const fp *)FROB1; k = t; }
    else if (t < 20) { src = (const fp *)FROB2; k = t - 10; }
    else if (t < 30) { src = (const fp *)FROB3; k = t - 20; }
    else if (t < 32) { src = (const fp *)&PSI_CX; k = t - 30; }
    else if (t < 34) { src = (const fp *)&PSI_CY; k = t - 32; }
    else if (t < 35) { src = &PSI2_CX; k = 0; }
    else { src = &FP_ONE; k = 0; }
    dst[t] = src[k];
}

// One warp per block; block b runs the program on instance b: in0 + b * s_in0, in1 + b * s_in1, out0 + b * s_out
// (strides in field elements; the per-batch tails launch one block with zero strides, the small-batch route one block
// per signature set).
// STREAM: the program contains STORE operations (streamed outputs, fpprog.hpp); a separate instantiation because the
// round loop is latency-bound to the instruction — the extra branch costs the programs that do not need it 10 %.
template <bool STREAM>
__device__ __forceinline__ void fp_program_body(const uint32_t *prog, const fp *in0, const fp *in1, const fp *cst, fp *out0,
                                                size_t s_in0, size_t s_in1, size_t s_out) {
    extern __shared__ uint4 sm4[];
    fp *slots = (fp *)sm4;
    const int lane = threadIdx.x;
    if (s_in0 != ~(size_t)0) {                             // ~0: the caller has positioned the pointers (k_fp_program_rows)
        in0 += (size_t)blockIdx.x * s_in0;
        if (in1) in1 += (size_t)blockIdx.x * s_in1;
        out0 += (size_t)blockIdx.x * s_out;
    }
    const uint32_t nr = prog[0], nin = prog[2], nout = prog[3];
    if (lane == 0) fp_set_zero(slots[0]);
    for (uint32_t e = lane; e < nin; e += 32) {
        uint32_t sl = prog[4 + 2 * e], ref = prog[5 + 2 * e], buf = ref >> 24, idx = ref & 0xffffffu;
        const fp *src = buf == 0 ? in0 : (buf == 1 ? in1 : cst);
        slots[sl] = src[idx];
    }
    __syncwarp();
    // operation words are prefetched four rounds ahead so that their global-memory latency overlaps the arithmetic
    const uint32_t *rp = prog + 4 + 2 * (nin + nout) + lane;
    uint32_t wq[4];
#pragma unroll
    for (int k = 0; k < 4; k++) wq[k] = (uint32_t)k < nr ? rp[32 * k] : 0u;
    for (uint32_t r = 0; r < nr; r += 4) {
#pragma unroll
        for (int k = 0; k < 4; k++) {
            const uint32_t w = wq[k];
            wq[k] = r + k + 4 < nr ? rp[32 * (r + k + 4)] : 0u;
            if (STREAM) {
                const uint32_t opc = w >> 30;
                if (opc) {
                    fp x = slots[(w >> 10) & 1023], y = slots[w & 1023], t;
                    if (opc == 1) fp_mul(t, x, y);
                    else if (opc == 2) fp_add(t, x, y);
                    else fp_sub(t, x, y);
                    slots[(w >> 20) & 1023] = t;
                } else if (w) {                           // STORE: a streamed output leaves its slot now
                    out0[(((w >> 20) & 1023) << 10) | (w & 1023)] = slots[(w >> 10) & 1023];
                }
            } else if (w) {
                fp x = slots[(w >> 10) & 1023], y = slots[w & 1023], t;
                const uint32_t opc = w >> 30;
                if (opc == 1) fp_mul(t, x, y);
                else if (opc == 2) fp_add(t, x, y);
                else fp_sub(t, x, y);
                slots[(w >> 20) & 1023] = t;
            }
            __syncwarp();
        }
    }
    const uint32_t *op = prog + 4 + 2 * nin;
    for (uint32_t e = lane; e < nout; e += 32) out0[op[2 * e + 1] & 0xffffffu] = slots[op[2 * e]];
}
__global__ void __launch_bounds__(32) k_fp_program(const uint32_t *prog, const fp *in0, const fp *in1, const fp *cst, fp *out0,
                                                   size_t s_in0, size_t s_in1, size_t s_out) {
    fp_program_body<false>(prog, in0, in1, cst, out0, s_in0, s_in1, s_out);
}
__global__ void __launch_bounds__(32) k_fp_program_stream(const uint32_t *prog, const fp *in0, const fp *in1, const fp *cst,
                                                          fp *out0, size_t s_in0, size_t s_in1, size_t s_out) {
    fp_program_body<true>(prog, in0, in1, cst, out0, s_in0, s_in1, s_out);
}

// ---- format 2 (fpprog.hpp compile2): rounds of products and rounds of linear combinations --------------------------
// A round is 32 x 16 bytes; a LIN lane evaluates sum_pos mag * slot - sum_neg mag * slot (mod p) over up to seven
// operands in one step (fplin.cuh), so the three to six addition levels that the tower formulas put between two
// levels of products are ONE round.  Lanes of a round all hold the same kind of operation (or a STORE / nothing).
template <bool STREAM>
__device__ __forceinline__ void fp_program2_body(const uint32_t *prog, const fp *in0, const fp *in1, const fp *cst, fp *out0,
                                                 size_t s_in0, size_t s_in1, size_t s_out) {
    extern __shared__ uint4 sm4[];
    fp *slots = (fp *)sm4;
    const int lane = threadIdx.x;
    if (s_in0 != ~(size_t)0) {
        in0 += (size_t)blockIdx.x * s_in0;
        if (in1) in1 += (size_t)blockIdx.x * s_in1;
        out0 += (size_t)blockIdx.x * s_out;
    }
    const uint32_t nr = prog[0], nin = prog[2], nout = prog[3];
    if (lane == 0) fp_set_zero(slots[0]);
    for (uint32_t e = lane; e < nin; e += 32) {
        uint32_t sl = prog[4 + 2 * e], ref = prog[5 + 2 * e], buf = ref >> 24, idx = ref & 0xffffffu;
        const fp *src = buf == 0 ? in0 : (buf == 1 ? in1 : cst);
        slots[sl] = src[idx];
    }
    __syncwarp();
    const uint4 *rp = (const uint4 *)(prog + ((4 + 2 * (nin + nout) + 3) & ~3u)) + lane;
    uint4 wq[4];
#pragma unroll
    for (int k = 0; k < 4; k++) wq[k] = (uint32_t)k < nr ? rp[32 * k] : make_uint4(0, 0, 0, 0);
    for (uint32_t r = 0; r < nr; r += 4) {
#pragma unroll
        for (int k = 0; k < 4; k++) {
            const uint4 w = wq[k];
            wq[k] = r + k + 4 < nr ? rp[32 * (r + k + 4)] : make_uint4(0, 0, 0, 0);
            const uint32_t op = w.x >> 30;
            if (__any_sync(0xffffffffu, op == 1)) {
                if (op == 1) {
                    fp x = slots[w.y & 1023], y = slots[(w.y >> 10) & 1023], t;
                    fp_mul(t, x, y);
                    slots[(w.x >> 20) & 1023] = t;
                }
            } else {
                const uint32_t npos = op == 2 ? (w.x >> 17) & 7 : 0, nneg = op == 2 ? (w.x >> 14) & 7 : 0;
                const uint32_t mp = __reduce_max_sync(0xffffffffu, npos), mn = __reduce_max_sync(0xffffffffu, nneg);
                if (__any_sync(0xffffffffu, op == 2)) {
                    const uint32_t t[7] = {w.y & 0x3fffu, (w.y >> 14) & 0x3fffu, w.z & 0x3fffu, (w.z >> 14) & 0x3fffu,
                                           w.w & 0x3fffu, (w.w >> 14) & 0x3fffu, w.x & 0x3fffu};
                    lin_acc A;
                    lin_clear(A);
#pragma unroll
                    for (int j = 0; j < 7; j++)
                        if ((uint32_t)j < mp) {                       // uniform: every lane walks the longest list of the round
                            const uint32_t code = (uint32_t)j < npos ? t[j] : 0u;
                            fp x = slots[code & 1023];
                            lin_add_term(A.P, x, code >> 10);
                        }
#pragma unroll
                    for (int j = 0; j < 7; j++)
                        if ((uint32_t)j < mn) {
                            const uint32_t code = (uint32_t)j < nneg ? t[6 - j] : 0u;
                            fp x = slots[code & 1023];
                            lin_add_term(A.N, x, code >> 10);
                        }
                    if (op == 2) {
                        fp rr;
                        lin_finish(rr, A);
                        slots[(w.x >> 20) & 1023] = rr;
                    }
                }
            }
            if (STREAM && op == 0 && w.x) out0[w.z] = slots[w.y];   // a streamed output leaves its slot now
            __syncwarp();
        }
    }
    const uint32_t *op = prog + 4 + 2 * nin;
    for (uint32_t e = lane; e < nout; e += 32) out0[op[2 * e + 1] & 0xffffffu] = slots[op[2 * e]];
}
__global__ void __launch_bounds__(32) k_fp_program2(const uint32_t *prog, const fp *in0, const fp *in1, const fp *cst, fp *out0,
                                                    size_t s_in0, size_t s_in1, size_t s_out) {
    fp_program2_body<false>(prog, in0, in1, cst, out0, s_in0, s_in1, s_out);
}
__global__ void __launch_bounds__(32) k_fp_program2_stream(const uint32_t *prog, const fp *in0, const fp *in1, const fp *cst,
                                                           fp *out0, size_t s_in0, size_t s_in1, size_t s_out) {
    fp_program2_body<true>(prog, in0, in1, cst, out0, s_in0, s_in1, s_out);
}
__global__ void __launch_bounds__(32) k_fp_program2_rows(const uint32_t *prog, const fp *in, const fp *cst, fp *out, unsigned m,
                                                         size_t in_stride, size_t out_stride) {
    const size_t j = blockIdx.x / m, g = blockIdx.x % m;
    fp_program2_body<false>(prog, in + (j * in_stride + 8 * g) * 12, nullptr, cst, out + (j * out_stride + g) * 12, ~(size_t)0, 0, 0);
}

// Row-wise instances for the product trees of the GT product: block b = (row j, group g) of m groups per row reads the 8
// Fp12 values in[j * in_stride + 8 g ..] and writes one to out[j * out_stride + g] (strides in Fp12 values).
__global__ void __launch_bounds__(32) k_fp_program_rows(const uint32_t *prog, const fp *in, const fp *cst, fp *out, unsigned m,
                                                        size_t in_stride, size_t out_stride) {
    const size_t j = blockIdx.x / m, g = blockIdx.x % m;
    fp_program_body<false>(prog, in + (j * in_stride + 8 * g) * 12, nullptr, cst, out + (j * out_stride + g) * 12, ~(size_t)0, 0, 0);
}

// the Fp inversion lifted out of the final-exponentiation program (fpprog.hpp INV_EXTERNAL): one thread, binary Euclid
__global__ void k_fp_inv_one(const fp *in, fp *out) {
    if (blockIdx.x != 0 || threadIdx.x != 0) return;
    fp a = *in, r;
    fp_inv_vartime(r, a);
    *out = r;
}

// verdict and canonical GT bytes of the final exponentiation result (fp12_tower.c:773-786): 12 lanes, one Fp each
__global__ void k_final_out(const fp12 *gt, int count, const int *flags, uint8_t *gt_bytes, int *is_one) {
    const int t = threadIdx.x;
    if (blockIdx.x != 0 || t >= 12) return;
    if (t == 0) {
        int bad = 0;
        if (flags) for (int i = 0; i < count; i++) bad |= flags[i];
        is_one[1] = bad;
        is_one[0] = fp12_is_one(*gt) ? 1 : 0;
    }
    // output order: for i in 0..2, j in 0..1: a[j][i].re || a[j][i].im  -> Fp number t = 4i + 2j + k reads c[3j+i].k
    const int i = t >> 2, j = (t >> 1) & 1, k = t & 1;
    const fp2 *c = &gt->c0.c0;
    fp v;
    fp_from_mont(v, k ? c[3 * j + i].c1 : c[3 * j + i].c0);
    uint8_t *out = gt_bytes + 48 * t;
    for (int b = 0; b < 48; b++) out[b] = (uint8_t)(v.l[(47 - b) >> 2] >> (8 * ((47 - b) & 3)));
}

// single-thread reference of the same tail (kept for BLSGPU_SERIAL_TAIL=1 cross-checks)
__global__ void k_final(const fp12 *partials, int count, const int *flags, uint8_t *gt_bytes, int *is_one) {
    if (blockIdx.x != 0 || threadIdx.x != 0) return;
    int bad = 0;
    if (flags) for (int i = 0; i < count; i++) bad |= flags[i];
    is_one[1] = bad;
    fp12 acc = partials[0];
    for (int i = 1; i < count; i++) { fp12 b = partials[i]; fp12_mul(acc, acc, b); }
    fp12 gt;
    final_exp(gt, acc);
    *is_one = fp12_is_one(gt) ? 1 : 0;
    fp12_to_bytes(gt_bytes, gt);
}

// ---- generic hash_to_G2 entry (arbitrary message length and DST, both in global memory) ----
// message i is msgs[offs[i] .. offs[i+1]) when offs is given, else msgs[i*msg_len .. (i+1)*msg_len)
__global__ void BLS_LB k_hash_to_g2(const uint8_t *msgs, size_t n, size_t msg_len, const uint32_t *offs, const uint8_t *dst,
                                    uint32_t dst_len, g2_aff *out_aff, uint8_t *out_comp) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    g2_jac h;
    if (offs) hash_to_g2_jac(h, msgs + offs[i], offs[i + 1] - offs[i], dst, dst_len);
    else hash_to_g2_jac(h, msgs + i * msg_len, msg_len, dst, dst_len);
    g2_aff a;
    pt_to_affine(a, h);
    if (out_aff) out_aff[i] = a;
    if (out_comp) g2_compress(out_comp + 96 * i, a);
}

// ---- aggregateVerify / fastAggregateVerify (SURVEY §8f N3; bls_sig_min_pubkey.nim:127-273) ----
// Pairs for the un-blinded check  FE( prod ML(pk_i, H(m_i)) * ML(sig, -G1) ) == 1: P[i] = pk_i (an infinite public key
// fails the call, aggregate.c:296), pair n = (sig, -G1); an infinite signature yields neutral lines (aggregate.c:486-492).
__global__ void k_verify_pairs(const g1_aff *pks, size_t n, const g2_aff *sig, g2_aff *Q, g1_aff *P, int *flags) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) {
        g1_aff pk = pks[i];
        if (aff_is_inf(pk)) atomicOr(flags, 1);
        P[i] = pk;
    } else if (i == n) {
        Q[n] = *sig;
        g1_aff g;
        g.x = G1_GEN_X;
        fp_neg(g.y, G1_GEN_Y);
        P[n] = g;
    }
}

// Segmented aggregateAll (blst_min_pubkey_sig_core.nim:179-195 once per segment): one warp per segment, every lane
// sums a strided slice with mixed additions, then a shared-memory tree over the 32 partial sums.
__global__ void __launch_bounds__(128) k_g1_seg_sum(const g1_aff *pts, const uint32_t *offs, size_t nseg, g1_jac *out) {
    __shared__ g1_jac sm[4][16];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const size_t sgm = (size_t)blockIdx.x * 4 + warp;
    if (sgm >= nseg) return;                               // whole warp leaves together
    const uint32_t lo = offs[sgm], hi = offs[sgm + 1];
    g1_jac acc;
    pt_set_inf(acc);
    for (uint32_t i = lo + lane; i < hi; i += 32) {
        g1_aff a = pts[i];
        pt_add_affine(acc, acc, a);
    }
    for (int half = 16; half >= 1; half >>= 1) {
        if (lane >= half && lane < 2 * half) sm[warp][lane - half] = acc;
        __syncwarp();
        if (lane < half) {
            g1_jac b = sm[warp][lane];
            pt_add(acc, acc, b);
        }
        __syncwarp();
    }
    if (lane == 0) out[sgm] = acc;
}
__global__ void BLS_LB k_g1_to_affine_many(const g1_jac *in, size_t n, g1_aff *out) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    g1_jac j = in[i];
    g1_aff a;
    pt_to_affine(a, j);
    out[i] = a;
}

// ---- batched fromBytes with checks (SURVEY §8f N2; io.cuh) ----
__global__ void BLS_LB k_pubkeys_from_bytes(const uint8_t *in, size_t n, int len, int group_check, g1_aff *out,
                                            uint8_t *status, int *nfail) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint8_t raw[96];
    for (int k = 0; k < len; k++) raw[k] = in[i * len + k];
    g1_aff p;
    int err = pubkey_from_bytes(p, raw, len, group_check != 0);
    out[i] = p;
    status[i] = (uint8_t)err;
    if (err) atomicAdd(nfail, 1);
}
__global__ void BLS_LB k_signatures_from_bytes(const uint8_t *in, size_t n, int len, int group_check, g2_aff *out,
                                               uint8_t *status, int *nfail) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint8_t raw[192];
    for (int k = 0; k < len; k++) raw[k] = in[i * len + k];
    g2_aff p;
    int err = signature_from_bytes(p, raw, len, group_check != 0);
    out[i] = p;
    status[i] = (uint8_t)err;
    if (err) atomicAdd(nfail, 1);
}
__global__ void k_g1_compress(const g1_aff *in, size_t n, uint8_t *out) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    g1_aff a = in[i];
    g1_compress(out + 48 * i, a);
}
__global__ void k_g2_compress(const g2_aff *in, size_t n, uint8_t *out) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    g2_aff a = in[i];
    g2_compress(out + 96 * i, a);
}

// ---- aggregateAll helpers ----
__global__ void __launch_bounds__(128) k_g1_load(const g1_aff *in, size_t n, g1_jac *out) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    g1_aff a = in[i];
    g1_jac j;
    pt_from_affine(j, a);
    out[i] = j;
}
__global__ void __launch_bounds__(128) k_g2_load(const g2_aff *in, size_t n, g2_jac *out) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    g2_aff a = in[i];
    g2_jac j;
    pt_from_affine(j, a);
    out[i] = j;
}
__global__ void k_g1_to_affine(const g1_jac *in, g1_aff *out) {
    if (blockIdx.x != 0 || threadIdx.x != 0) return;
    g1_jac j = *in;
    g1_aff a;
    pt_to_affine_vt(a, j);
    *out = a;
}
__global__ void k_g2_to_affine(const g2_jac *in, g2_aff *out) {
    if (blockIdx.x != 0 || threadIdx.x != 0) return;
    g2_jac j = *in;
    g2_aff a;
    pt_to_affine_vt(a, j);
    *out = a;
}

// subtractAll (blst_min_pubkey_sig_core.nim:197-209): blst_p{1,2}_cneg of one Jacobian point in place.
template <class F> __global__ void k_pt_neg(jac_t<F> *p) {
    if (blockIdx.x != 0 || threadIdx.x != 0) return;
    jac_t<F> a = *p, r;
    pt_neg(r, a);
    *p = r;
}

// ---- diagnostics: the field primitives one at a time (blsgpu_test_field, blsgpu_test_fp) ----
// Records: nin field elements and nin_w u32 words in, nout elements and nout_w words out (words padded to 16 bytes).
// Geometry: a thread per record; a lane pair per record (fp2h.cuh, pair-uniform bounds check); one lane of a six-lane
// team per record or one team per record (launch shape of k_miller_acc_team: ACC_BS threads, ACC_TPW teams per warp).
enum { TF_THREAD, TF_PAIR, TF_TEAM_LANE, TF_TEAM };
struct test_field_shape { int nin, nin_w, nout, nout_w, geom; };
static const test_field_shape TEST_FIELD_OPS[BLSGPU_TF_COUNT] = {
    {2, 0, 1, 0, TF_THREAD}, {2, 0, 1, 0, TF_THREAD}, {1, 0, 1, 0, TF_THREAD}, {1, 0, 1, 0, TF_THREAD},   // mul .. sqr_ni
    {2, 0, 1, 0, TF_THREAD}, {2, 0, 1, 0, TF_THREAD}, {1, 0, 1, 0, TF_THREAD}, {1, 0, 1, 0, TF_THREAD},   // add .. inv
    {1, 0, 1, 0, TF_THREAD}, {1, 0, 1, 0, TF_THREAD}, {1, 0, 1, 0, TF_THREAD},                            // .. from_mont
    {1, 0, 0, 1, TF_THREAD}, {1, 0, 0, 1, TF_THREAD},                                                     // parity, lex
    {4, 0, 2, 0, TF_THREAD}, {2, 0, 2, 0, TF_THREAD}, {2, 0, 2, 0, TF_THREAD}, {3, 0, 2, 0, TF_THREAD},   // fp2 mul .. mul_fp
    {2, 0, 2, 0, TF_THREAD}, {2, 0, 2, 0, TF_THREAD}, {2, 0, 2, 1, TF_THREAD},                            // inv, inv_vt, rsqrt
    {2, 0, 0, 1, TF_THREAD}, {2, 0, 0, 1, TF_THREAD},                                                     // sgn0, lex
    {4, 0, 2, 0, TF_PAIR}, {2, 0, 2, 0, TF_PAIR}, {2, 0, 2, 0, TF_PAIR}, {3, 0, 2, 0, TF_PAIR},           // h_mul .. h_mul_fp
    {2, 0, 2, 0, TF_PAIR}, {2, 0, 2, 0, TF_PAIR},                                                         // h_conj, h_inv
    {6, 0, 1, 0, TF_TEAM_LANE}, {8, 2, 1, 0, TF_TEAM_LANE}, {18, 0, 12, 0, TF_TEAM}, {12, 0, 12, 0, TF_TEAM},
    {14, 14, 1, 0, TF_THREAD},                                                                            // lin_finish
};
static inline size_t test_field_rec(int nfe, int nw) { return 48 * (size_t)nfe + 16 * (((size_t)nw + 3) / 4); }

__global__ void __launch_bounds__(ACC_BS) k_test_field(int op, const uint8_t *in, size_t in_rec, size_t n, uint8_t *out,
                                                      size_t out_rec) {
    __shared__ acc_team_sm sm[ACC_TPB];
    const int tid = threadIdx.x;
    if (op >= BLSGPU_TF_TEAM_DOT3 && op <= BLSGPU_TF_TEAM_SQUARE) {
        const int lane = tid & 31, warp = tid >> 5;
        if (lane >= 6 * ACC_TPW) return;                   // lanes 30, 31 idle, as in k_miller_acc_team
        const uint32_t mask = (1u << (6 * ACC_TPW)) - 1;
        const int team = lane / 6, k = lane % 6;
        acc_team_sm &T = sm[warp * ACC_TPW + team];
        const size_t g = ((size_t)blockIdx.x * (ACC_BS / 32) + warp) * ACC_TPW + team;
        if (op == BLSGPU_TF_TEAM_DOT3 || op == BLSGPU_TF_TEAM_DOT4) {
            const size_t i = 6 * g + k;                    // a record per lane; no barriers on this path
            if (i >= n) return;
            const fp *x = (const fp *)(in + i * in_rec);
            fp *S = (fp *)&T + 4 * k;                      // streamed side from shared memory, register side from the record
            fp r;
            if (op == BLSGPU_TF_TEAM_DOT3) {
                for (int t = 0; t < 3; t++) S[t] = x[3 + t];
                team_dot3(r, &x[0], &x[1], &x[2], &S[0], &S[1], &S[2]);
            } else {
                const uint32_t *w = (const uint32_t *)(x + 8);
                for (int t = 0; t < 4; t++) S[t] = x[4 + t];
                const fp *const ap[4] = {&x[0], &x[1], &x[2], &x[3]}, *const bp[4] = {&S[0], &S[1], &S[2], &S[3]};
                team_dot4(r, ap, bp, w[0], w[1]);
            }
            *(fp *)(out + i * out_rec) = r;
            return;
        }
        // a record per team: Fp12 f in the tower layout (coefficient of w^k at Fp2 index 3 (k & 1) + (k >> 1)), then
        // the line; teams past n run on zeros so that every lane of the mask reaches every barrier
        const bool valid = g < n;
        const fp *x = (const fp *)(in + (valid ? g : 0) * in_rec);
        const int s = 3 * (k & 1) + (k >> 1);
        fp c0, c1;
        if (valid) { c0 = x[2 * s]; c1 = x[2 * s + 1]; } else { fp_set_zero(c0); fp_set_zero(c1); }
        team_store_coeff(T, k, c0, c1);
        if (op == BLSGPU_TF_TEAM_MUL_LINE) {
            fp v;
            if (valid) v = x[12 + k]; else fp_set_zero(v);
            T.l[k] = v;
            __syncwarp(mask);
            if (k < 3) { fp sum; fp_add(sum, T.l[2 * k], T.l[2 * k + 1]); T.l[6 + k] = sum; }
            __syncwarp(mask);
            team_mul_line(T, k, mask);
        } else {
            __syncwarp(mask);
            team_square(T, k, mask);
        }
        if (valid) {
            fp *y = (fp *)(out + g * out_rec);
            y[2 * s] = T.f[k][FV_C0];
            y[2 * s + 1] = T.f[k][FV_C1];
        }
        return;
    }
    if (op >= BLSGPU_TF_H_MUL && op <= BLSGPU_TF_H_INV) {
        const size_t e = ((size_t)blockIdx.x * blockDim.x + tid) >> 1;
        if (e >= n) return;                                // the same for both lanes of a pair
        const fp *x = (const fp *)(in + e * in_rec);
        const int h = tid & 1;
        fp2h a, b, r;
        a.v = x[h];
        switch (op) {
            case BLSGPU_TF_H_MUL: b.v = x[2 + h]; h_mul(r, a, b); break;
            case BLSGPU_TF_H_SQR: h_sqr(r, a); break;
            case BLSGPU_TF_H_MUL_XI: h_mul_xi(r, a); break;
            case BLSGPU_TF_H_MUL_FP: { fp kk = x[2]; h_mul_fp(r, a, kk); break; }
            case BLSGPU_TF_H_CONJ: h_conj(r, a); break;
            default: h_inv(r, a); break;
        }
        ((fp *)(out + e * out_rec))[h] = r.v;
        return;
    }
    const size_t i = (size_t)blockIdx.x * blockDim.x + tid;
    if (i >= n) return;
    const fp *x = (const fp *)(in + i * in_rec);
    fp *y = (fp *)(out + i * out_rec);
    const fp a = x[0];
    fp r;
    fp2 a2, r2;
    if (op >= BLSGPU_TF_FP2_MUL && op <= BLSGPU_TF_FP2_IS_LEXICALLY_LARGEST) { a2.c0 = x[0]; a2.c1 = x[1]; }
    switch (op) {
        case BLSGPU_TF_FP_MUL: { fp b = x[1]; fp_mul(r, a, b); break; }
        case BLSGPU_TF_FP_MUL_NI: fp_mul_ni(r, a, x[1]); break;
        case BLSGPU_TF_FP_SQR: fp_sqr(r, a); break;
        case BLSGPU_TF_FP_SQR_NI: fp_sqr_ni(r, a); break;
        case BLSGPU_TF_FP_ADD: { fp b = x[1]; fp_add(r, a, b); break; }
        case BLSGPU_TF_FP_SUB: { fp b = x[1]; fp_sub(r, a, b); break; }
        case BLSGPU_TF_FP_NEG: fp_neg(r, a); break;
        case BLSGPU_TF_FP_INV: fp_inv(r, a); break;
        case BLSGPU_TF_FP_INV_VARTIME: fp_inv_vartime(r, a); break;
        case BLSGPU_TF_FP_POW_P34: fp_pow_p34(r, a); break;
        case BLSGPU_TF_FP_FROM_MONT: fp_from_mont(r, a); break;
        case BLSGPU_TF_FP_PARITY: *(uint32_t *)y = fp_parity(a); return;
        case BLSGPU_TF_FP_IS_LEXICALLY_LARGEST_CANON: *(uint32_t *)y = fp_is_lexically_largest_canon(a); return;
        case BLSGPU_TF_FP2_MUL: { fp2 b2; b2.c0 = x[2]; b2.c1 = x[3]; fp2_mul(r2, a2, b2); break; }
        case BLSGPU_TF_FP2_SQR: fp2_sqr(r2, a2); break;
        case BLSGPU_TF_FP2_MUL_XI: fp2_mul_xi(r2, a2); break;
        case BLSGPU_TF_FP2_MUL_FP: { fp kk = x[2]; fp2_mul_fp(r2, a2, kk); break; }
        case BLSGPU_TF_FP2_INV: fp2_inv(r2, a2); break;
        case BLSGPU_TF_FP2_INV_VARTIME: fp2_inv_vartime(r2, a2); break;
        case BLSGPU_TF_FP2_RSQRT_OR_Z: ((uint32_t *)(y + 2))[0] = fp2_rsqrt_or_z(r2, a2); break;
        case BLSGPU_TF_FP2_SGN0: *(uint32_t *)y = fp2_sgn0(a2); return;
        case BLSGPU_TF_FP2_IS_LEXICALLY_LARGEST: *(uint32_t *)y = fp2_is_lexically_largest(a2); return;
        default: {                                         // BLSGPU_TF_LIN_FINISH, built as fp_program2_body builds it
            const uint32_t *w = (const uint32_t *)(x + 14);
            lin_acc A;
            lin_clear(A);
            for (int j = 0; j < 7; j++) { fp t = x[j]; lin_add_term(A.P, t, w[j]); }
            for (int j = 0; j < 7; j++) { fp t = x[7 + j]; lin_add_term(A.N, t, w[7 + j]); }
            lin_finish(r, A);
            break;
        }
    }
    if (op >= BLSGPU_TF_FP2_MUL && op <= BLSGPU_TF_FP2_IS_LEXICALLY_LARGEST) { y[0] = r2.c0; y[1] = r2.c1; }
    else y[0] = r;
}

// Integer-multiply pipe peak: 8 independent mad.wide (or mad.lo) chains per thread, no memory traffic.
template <int WIDE>
__global__ void __launch_bounds__(256) k_imad_peak(uint32_t *sink, int iters, uint32_t seed) {
    uint32_t a = seed + threadIdx.x, b = seed * 3 + blockIdx.x;
    if (WIDE) {
        uint64_t acc[8];
        for (int k = 0; k < 8; k++) acc[k] = k;
        for (int i = 0; i < iters; i++) {
#pragma unroll
            for (int u = 0; u < 8; u++) {
#pragma unroll
                for (int k = 0; k < 8; k++)
                    asm volatile("mad.wide.u32 %0, %1, %2, %0;" : "+l"(acc[k]) : "r"(a + k), "r"(b + u));
            }
        }
        uint64_t s = 0;
        for (int k = 0; k < 8; k++) s ^= acc[k];
        if (s == 0x1234567) sink[0] = (uint32_t)s;
    } else {
        uint32_t acc[8];
        for (int k = 0; k < 8; k++) acc[k] = k;
        for (int i = 0; i < iters; i++) {
#pragma unroll
            for (int u = 0; u < 8; u++) {
#pragma unroll
                for (int k = 0; k < 8; k++)
                    asm volatile("mad.lo.u32 %0, %1, %2, %0;" : "+r"(acc[k]) : "r"(a + k), "r"(b + u));
            }
        }
        uint32_t s = 0;
        for (int k = 0; k < 8; k++) s ^= acc[k];
        if (s == 0x1234567) sink[0] = s;
    }
}

// Register-resident Fp multiplication throughput (ceiling of this fp_mul implementation): every thread runs a
// dependent chain x <- x*y, y <- y*x with no memory traffic.
__global__ void k_fpmul_peak(fp *sink, int iters, uint32_t seed) {
    fp x, y;
#pragma unroll
    for (int i = 0; i < 12; i++) { x.l[i] = seed + i + threadIdx.x; y.l[i] = seed * 7 + i + blockIdx.x; }
    x.l[11] &= 0x0fffffffu;
    y.l[11] &= 0x0fffffffu;
    for (int i = 0; i < iters; i++) {
        fp_mul(x, x, y);
        fp_mul(y, y, x);
    }
    if (x.l[0] == 0x12345 && y.l[3] == 0x54321) sink[0] = x;
}

// Synthetic valid signature sets, generated on the device (benchmark input only).
__global__ void BLS_LB k_make_sets(words8 seed, size_t first, size_t n, sigset *out) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint64_t idx = first + i;
    // sk = 1 + (SHA256(seed || LE64(idx)) mod 2^250)
    uint32_t h[8] = {0x6a09e667u, 0xbb67ae85u, 0x3c6ef372u, 0xa54ff53au, 0x510e527fu, 0x9b05688cu, 0x1f83d9abu, 0x5be0cd19u};
    uint32_t w[16];
    for (int k = 0; k < 8; k++) w[k] = seed.w[k];
    w[8] = __byte_perm((uint32_t)idx, 0, 0x0123);
    w[9] = __byte_perm((uint32_t)(idx >> 32), 0, 0x0123);
    w[10] = 0x80000000u;
    for (int k = 11; k < 15; k++) w[k] = 0;
    w[15] = 320;
    sha256_block(h, w);
    uint32_t sk[8];
    for (int k = 0; k < 8; k++) sk[k] = h[7 - k];
    sk[7] &= 0x03ffffffu;
    sk[0] |= 1;                                         // non-zero
    // msg = SHA256("blsgpu" || LE64(idx))
    uint8_t pre[14] = {'b', 'l', 's', 'g', 'p', 'u'};
    for (int k = 0; k < 8; k++) pre[6 + k] = (uint8_t)(idx >> (8 * k));
    sha256_ctx c;
    sha256_init(c);
    sha256_update(c, pre, 14);
    uint32_t md[8];
    sha256_final(c, md);
    uint8_t msg[32], dst[43];
    for (int k = 0; k < 32; k++) msg[k] = (uint8_t)(md[k >> 2] >> (24 - 8 * (k & 3)));
    for (int k = 0; k < 43; k++) dst[k] = DST_ETH2[k];
    g1_jac g, pkj;
    g.x = G1_GEN_X; g.y = G1_GEN_Y; g.z = FP_ONE;
    pt_mul_words(pkj, g, sk, 8);
    g2_jac hj, sj;
    hash_to_g2_jac(hj, msg, 32, dst, 43);
    pt_mul_words(sj, hj, sk, 8);
    sigset s;
    pt_to_affine(s.pk, pkj);
    pt_to_affine(s.sig, sj);
    for (int k = 0; k < 32; k++) s.msg[k] = msg[k];
    out[i] = s;
}

}  // namespace bls
