// msm.cuh — multi-scalar multiplication in G1 and G2: signed-digit Pippenger with a sorted bucket scatter.
// Restates the results of blst_p1s_mult_pippenger / blst_p2s_mult_pippenger (vendor/blst/src/multi_scalar.c:415-446;
// window loop :370-397, tile :332-368, bucket integration :295-311) — the affine sum  sum_i [k_i] P_i  is canonical,
// so the GPU decomposition is free to differ:
//   1. k_msm_count    signed window digits (Booth-style carry, digits in (-2^(c-1), 2^(c-1)]), histogram
//                     of (window, |digit|) with global atomics
//   2. k_msm_scan_*   exclusive prefix sums of the histogram and of the non-empty flags (three launches)
//   3. k_msm_scatter  counting-sort scatter of (point index, sign) into bucket order
//   4. k_msm_chunks   one thread per CHUNK = K consecutive entries of the sorted list, whatever buckets they fall in:
//                     gathers its points, mixed Jacobian additions, one partial per (chunk, bucket) run - every lane
//                     does exactly K additions, so neither a skewed digit distribution nor the spread of bucket
//                     sizes idles lanes
//   5. k_msm_combine  one thread per bucket sums its partials; buckets with more than MSM_BIG partials are
//                     deferred to k_msm_combine_big (one warp per bucket, shuffle tree)
//   6. k_msm_segment  running-sum integration of L-bucket segments, weighted by the segment base
//   7. k_tree_rows    per-window tree sum of the segment results
//   8. k_msm_horner   Horner over windows (c doublings each), Jacobian and/or affine output
// The same kernels serve the batch verifier's sum  S = sum_i [r_i] sig_i  (G2, 64-bit scalars, points read in place
// from the SignatureSet array) — vendor/blst/src/aggregate.c:321-335 accumulates that sum one scalar
// multiplication at a time.
// Scalars are NOT reduced mod r (as in the reference); the nbits low bits of each little-endian scalar are used.
#pragma once
#include <functional>
#include <string>
#include <type_traits>
#include "kernels.cuh"
#include "route.hpp"

namespace bls {

struct msm_state {
    uint8_t *buf = nullptr;
    size_t bytes = 0;
    int sms = 148;                 // SM count of the device (B200: 148); set at context creation
    // window-group pipelining: the latency-bound tail of a group (combine, segment, tree, Horner) runs on this
    // higher-priority stream underneath the bucket accumulation of the next group
    cudaStream_t tail = nullptr;
    cudaEvent_t ev_group[8] = {}, ev_done = nullptr;
    bool ev_ok = false;
};

static inline void msm_free(msm_state &m) {
    if (m.ev_ok) { for (int i = 0; i < 8; i++) cudaEventDestroy(m.ev_group[i]); cudaEventDestroy(m.ev_done); m.ev_ok = false; }
    if (m.tail) { cudaStreamDestroy(m.tail); m.tail = nullptr; }
    if (m.buf) cudaFree(m.buf);
    m.buf = nullptr;
    m.bytes = 0;
}

// partials per bucket beyond which the block-wide combine takes over (measured: 8 beats 32 by 1.7 ms for the 4 096-set
// signature sum, where every bucket holds ~32 partials, and costs nothing at 2^20 points; 4 floods the big-bucket path)
#ifndef MSM_BIG
#define MSM_BIG 8
#endif

// signed digit of window w (width c) of the nbits-bit little-endian scalar at sc (sb bytes)
__device__ __forceinline__ int msm_digit(const uint8_t *sc, int sb, int nbits, int c, int w, int &carry) {
    int bit = w * c;
    uint32_t raw = 0;
    // gather c bits starting at `bit`, masking everything at or above nbits
    for (int k = 0; k < c; k += 8) {
        int b0 = bit + k;
        if (b0 >= nbits) break;
        int byte = b0 >> 3, sh = b0 & 7;
        uint32_t v = sc[byte];
        if (byte + 1 < sb) v |= (uint32_t)sc[byte + 1] << 8;
        v >>= sh;
        int take = c - k < 8 ? c - k : 8;
        if (b0 + take > nbits) take = nbits - b0;
        v &= (1u << take) - 1;
        raw |= v << k;
    }
    int d = (int)raw + carry;
    if (d > (1 << (c - 1))) { d -= (1 << c); carry = 1; } else carry = 0;
    return d;
}

__global__ void __launch_bounds__(256) k_msm_count(const uint8_t *scalars, size_t sstride, size_t n, int sb, int nbits, int c,
                                                   int nwin, uint32_t *counts) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint8_t *sc = scalars + i * sstride;
    int carry = 0;
    const uint32_t B = 1u << (c - 1);
    for (int w = 0; w < nwin; w++) {
        int d = msm_digit(sc, sb, nbits, c, w, carry);
        if (d != 0) atomicAdd(&counts[(size_t)w * B + (uint32_t)(d < 0 ? -d : d) - 1], 1u);
    }
}

// Exclusive scans over the m buckets, three launches (block sums -> scan of the block sums -> apply):
//   offsets[0..m] of the entry counts (cursor = a working copy for the scatter), rank[0..m] of [count > 0]
//   (rank[b] = number of non-empty buckets before b; it places the partial sums, see k_msm_chunks).
__device__ __forceinline__ void msm_block_scan2(uint32_t v0, uint32_t v1, uint32_t &x0, uint32_t &x1, uint32_t &t0, uint32_t &t1,
                                                uint32_t (*ws)[32]) {
    // inclusive scans x0/x1 of v0/v1 over the 1024 threads of the block, block totals in t0/t1
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    x0 = v0; x1 = v1;
    for (int o = 1; o < 32; o <<= 1) {
        uint32_t y0 = __shfl_up_sync(0xffffffffu, x0, o), y1 = __shfl_up_sync(0xffffffffu, x1, o);
        if (lane >= o) { x0 += y0; x1 += y1; }
    }
    if (lane == 31) { ws[0][wid] = x0; ws[1][wid] = x1; }
    __syncthreads();
    if (wid < 2) {
        uint32_t s = ws[wid][lane], t = s;
        for (int o = 1; o < 32; o <<= 1) {
            uint32_t y = __shfl_up_sync(0xffffffffu, t, o);
            if (lane >= o) t += y;
        }
        ws[wid][lane] = t - s;            // exclusive warp offsets
        if (lane == 31) ws[2 + wid][0] = t;
    }
    __syncthreads();
    x0 += ws[0][wid];
    x1 += ws[1][wid];
    t0 = ws[2][0];
    t1 = ws[3][0];
}

__global__ void __launch_bounds__(1024) k_msm_scan_blocks(const uint32_t *counts, size_t m, uint32_t *bsums) {
    __shared__ uint32_t ws[4][32];
    size_t i = (size_t)blockIdx.x * 1024 + threadIdx.x;
    uint32_t v0 = i < m ? counts[i] : 0, v1 = v0 ? 1u : 0u, x0, x1, t0, t1;
    msm_block_scan2(v0, v1, x0, x1, t0, t1, ws);
    if (threadIdx.x == 0) { bsums[2 * blockIdx.x] = t0; bsums[2 * blockIdx.x + 1] = t1; }
}

// in-place exclusive scan of the nblk (entries, non-empty) pairs; one block
__global__ void __launch_bounds__(1024) k_msm_scan_top(uint32_t *bsums, size_t nblk) {
    __shared__ uint32_t ws[4][32];
    __shared__ uint32_t carry_s[2];
    if (threadIdx.x < 2) carry_s[threadIdx.x] = 0;
    __syncthreads();
    for (size_t base = 0; base < nblk; base += 1024) {
        size_t i = base + threadIdx.x;
        uint32_t v0 = i < nblk ? bsums[2 * i] : 0, v1 = i < nblk ? bsums[2 * i + 1] : 0, x0, x1, t0, t1;
        msm_block_scan2(v0, v1, x0, x1, t0, t1, ws);
        uint32_t c0 = carry_s[0], c1 = carry_s[1];
        if (i < nblk) { bsums[2 * i] = c0 + x0 - v0; bsums[2 * i + 1] = c1 + x1 - v1; }
        __syncthreads();
        if (threadIdx.x == 0) { carry_s[0] = c0 + t0; carry_s[1] = c1 + t1; }
        __syncthreads();
    }
}

__global__ void __launch_bounds__(1024) k_msm_scan_apply(const uint32_t *counts, size_t m, const uint32_t *bsums,
                                                         uint32_t *offsets, uint32_t *cursor, uint32_t *rank) {
    __shared__ uint32_t ws[4][32];
    size_t i = (size_t)blockIdx.x * 1024 + threadIdx.x;
    uint32_t v0 = i < m ? counts[i] : 0, v1 = v0 ? 1u : 0u, x0, x1, t0, t1;
    msm_block_scan2(v0, v1, x0, x1, t0, t1, ws);
    uint32_t e0 = bsums[2 * blockIdx.x] + x0 - v0, e1 = bsums[2 * blockIdx.x + 1] + x1 - v1;
    if (i < m) { offsets[i] = e0; cursor[i] = e0; rank[i] = e1; }
    if (i == m - 1) { offsets[m] = e0 + v0; rank[m] = e1 + v1; }
}

__global__ void __launch_bounds__(256) k_msm_scatter(const uint8_t *scalars, size_t sstride, size_t n, int sb, int nbits, int c,
                                                     int nwin, uint32_t *cursor, uint32_t *entries) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint8_t *sc = scalars + i * sstride;
    int carry = 0;
    const uint32_t B = 1u << (c - 1);
    for (int w = 0; w < nwin; w++) {
        int d = msm_digit(sc, sb, nbits, c, w, carry);
        if (d != 0) {
            uint32_t pos = atomicAdd(&cursor[(size_t)w * B + (uint32_t)(d < 0 ? -d : d) - 1], 1u);
            entries[pos] = ((uint32_t)i << 1) | (d < 0 ? 1u : 0u);
        }
    }
}

// Chunk t sums entries [t*K, (t+1)*K) of the bucket-sorted entry list: every lane of a warp performs exactly K mixed
// additions whatever the digit distribution (no idle lanes, no serialisation on a heavy bucket).  A run of one bucket
// inside a chunk yields one partial, stored at slot t + rank[b]: slots increase strictly along the (chunk, bucket) run
// sequence, and the partials of bucket b are the contiguous slots t0 + rank[b] .. t1 + rank[b] for the chunks t0..t1
// its entries touch.
template <class F>
__global__ void BLS_LB k_msm_chunks(const uint8_t *points, size_t pstride, const uint32_t *offsets, const uint32_t *rank,
                                    const uint32_t *entries, size_t b0, size_t b1, uint32_t K, jac_t<F> *partials) {
    // window group = buckets [b0, b1): its entries are [S, E); chunks, partial slots and ranks are group-relative
    const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t S = offsets[b0], E = offsets[b1], rank0 = rank[b0];
    if (t * K >= (size_t)(E - S)) return;
    const uint32_t e0 = S + (uint32_t)(t * K), e1 = E - e0 > K ? e0 + K : E;
    size_t lo = b0, hi = b1;                       // largest b with offsets[b] <= e0: the (non-empty) bucket of entry e0
    while (hi - lo > 1) {
        size_t mid = (lo + hi) >> 1;
        if (offsets[mid] <= e0) lo = mid; else hi = mid;
    }
    size_t b = lo;
    uint32_t bend = offsets[b + 1];
    jac_t<F> acc;
    pt_set_inf(acc);
    for (uint32_t e = e0; e < e1; e++) {
        if (e == bend) {                           // bucket boundary: flush the run, move to the next non-empty bucket
            partials[t + (rank[b] - rank0)] = acc;
            pt_set_inf(acc);
            do { b++; bend = offsets[b + 1]; } while (bend <= e);
        }
        uint32_t ent = entries[e];
        aff_t<F> p = *(const aff_t<F> *)(points + (size_t)(ent >> 1) * pstride);
        if (ent & 1) f_neg(p.y, p.y);
        pt_add_affine(acc, acc, p);
    }
    partials[t + (rank[b] - rank0)] = acc;
}

// partial slots of bucket b (count > 0): [base, base + np)
__device__ __forceinline__ void msm_bucket_slots(const uint32_t *offsets, const uint32_t *rank, size_t b, uint32_t K,
                                                 uint32_t S, uint32_t rank0, uint32_t &base, uint32_t &np) {
    const uint32_t o0 = offsets[b], o1 = offsets[b + 1];
    if (o1 == o0) { base = 0; np = 0; return; }
    const uint32_t t0 = (o0 - S) / K, t1 = (o1 - 1 - S) / K;
    base = t0 + (rank[b] - rank0);
    np = t1 - t0 + 1;
}

template <class F>
__global__ void BLS_LB k_msm_combine(const jac_t<F> *partials, const uint32_t *offsets, const uint32_t *rank, size_t b0,
                                     size_t b1, uint32_t K, jac_t<F> *buckets, uint32_t *biglist, uint32_t *bigcount) {
    size_t b = b0 + (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= b1) return;
    uint32_t base, np;
    msm_bucket_slots(offsets, rank, b, K, offsets[b0], rank[b0], base, np);
    if (np > MSM_BIG) {
        biglist[b0 + atomicAdd(bigcount, 1u)] = (uint32_t)b;
        return;
    }
    jac_t<F> acc;
    pt_set_inf(acc);
    if (np) acc = partials[base];
    for (uint32_t t = 1; t < np; t++) {
        jac_t<F> x = partials[base + t];
        pt_add(acc, acc, x);
    }
    buckets[b] = acc;
}

// one BLOCK per over-full bucket: the 128 threads stride over its partials, a shuffle tree per warp, then the four
// warp sums through shared memory.  (A window whose digits take only a few values — a short top window, or scalars
// that are all equal — puts n / K partials into one bucket; 128 lanes keep that a few dozen serial additions.)
template <class F>
__global__ void BLS_LB k_msm_combine_big(const jac_t<F> *partials, const uint32_t *offsets, const uint32_t *rank, size_t b0,
                                         uint32_t K, const uint32_t *biglist, const uint32_t *bigcount, jac_t<F> *buckets) {
    __shared__ jac_t<F> wsum[4];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const uint32_t nbig = *bigcount;
    for (uint32_t i = blockIdx.x; i < nbig; i += gridDim.x) {
        const uint32_t b = biglist[b0 + i];
        uint32_t base, np;
        msm_bucket_slots(offsets, rank, b, K, offsets[b0], rank[b0], base, np);
        jac_t<F> acc;
        pt_set_inf(acc);
        for (uint32_t t = threadIdx.x; t < np; t += blockDim.x) {
            jac_t<F> x = partials[base + t];
            pt_add(acc, acc, x);
        }
        for (int o = 16; o >= 1; o >>= 1) {
            jac_t<F> other;
            uint32_t *dst = (uint32_t *)&other;
            const uint32_t *src = (const uint32_t *)&acc;
            for (int k = 0; k < (int)(sizeof(jac_t<F>) / 4); k++) dst[k] = __shfl_down_sync(0xffffffffu, src[k], o);
            pt_add(acc, acc, other);
        }
        if (lane == 0) wsum[wid] = acc;
        __syncthreads();
        if (threadIdx.x == 0) {
            for (int w = 1; w < 4; w++) { jac_t<F> x = wsum[w]; pt_add(acc, acc, x); }
            buckets[b] = acc;
        }
        __syncthreads();
    }
}

// segment j of window w covers digit magnitudes b in [j*L+1, j*L+L] (bucket index b-1):
//   T = sum_b (b - j*L) B_b  +  [j*L] sum_b B_b
template <class F>
__global__ void BLS_LB k_msm_segment(const jac_t<F> *buckets, int c, int nwin, uint32_t L, jac_t<F> *segs) {
    const uint32_t B = 1u << (c - 1);
    const uint32_t nseg = B / L;
    size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= (size_t)nwin * nseg) return;
    uint32_t w = (uint32_t)(t / nseg), j = (uint32_t)(t % nseg);
    const jac_t<F> *bk = buckets + (size_t)w * B + (size_t)j * L;
    jac_t<F> running, acc;
    pt_set_inf(running);
    pt_set_inf(acc);
    for (int b = (int)L - 1; b >= 0; b--) {
        jac_t<F> x = bk[b];
        pt_add(running, running, x);
        pt_add(acc, acc, running);
    }
    uint32_t k = j * L;
    if (k) {
        jac_t<F> m;
        pt_mul_words(m, running, &k, 1);
        pt_add(acc, acc, m);
    }
    segs[t] = acc;
}

// row-wise pairwise tree step over `rows` rows of `stride` entries
template <class F>
__global__ void BLS_LB k_tree_rows(jac_t<F> *S, int rows, size_t stride, size_t m, size_t half) {
    size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= (size_t)rows * half) return;
    size_t r = t / half, i = t % half;
    if (i + half >= m) return;
    jac_t<F> a = S[r * stride + i], b = S[r * stride + i + half];
    pt_add(a, a, b);
    S[r * stride + i] = a;
}

// Horner over the windows of one group, top window first: acc = [2^c] acc + W_w.  `carry` holds the running value
// across groups (read unless `first`, written unless this is the last group, which emits the result instead).
template <class F>
__global__ void k_msm_horner(const jac_t<F> *W, size_t stride, int nwin, int c, int first, int last, jac_t<F> *carry,
                             jac_t<F> *out_jac, aff_t<F> *out_aff) {
    if (blockIdx.x != 0 || threadIdx.x != 0) return;
    jac_t<F> acc;
    int w = nwin - 1;
    if (first) { acc = W[(size_t)w * stride]; w--; } else acc = *carry;
    for (; w >= 0; w--) {
        for (int k = 0; k < c; k++) pt_dbl(acc, acc);
        jac_t<F> x = W[(size_t)w * stride];
        pt_add(acc, acc, x);
    }
    if (!last) { *carry = acc; return; }
    if (out_jac) *out_jac = acc;
    if (out_aff) {
        aff_t<F> a;
        pt_to_affine_vt(a, acc);
        *out_aff = a;
    }
}

// G1 window Horner as a warp-cooperative dataflow program (fpprog.hpp build_msm_horner_g1, run by k_fp_program):
// the 255 sequential doublings cost two multiplication levels each instead of seven dependent multiplications.
// prep: window sums, Jacobian (X, Y, Z) -> homogeneous (X Z : Y : Z^3), infinity -> (0 : 1 : 0)
__global__ void k_msm_horner_prep(const g1_jac *W, size_t stride, int nwin, fp *hom) {
    const int w = blockIdx.x * blockDim.x + threadIdx.x;
    if (w >= nwin) return;
    g1_jac p = W[(size_t)w * stride];
    fp x, y, z;
    if (pt_is_inf(p)) {
        fp_set_zero(x); y = FP_ONE; fp_set_zero(z);
    } else {
        fp z2;
        fp_mul_ni(x, p.x, p.z);
        y = p.y;
        fp_sqr_ni(z2, p.z);
        fp_mul_ni(z, z2, p.z);
    }
    hom[3 * w] = x; hom[3 * w + 1] = y; hom[3 * w + 2] = z;
}
// finish: homogeneous (X : Y : Z) -> affine (X/Z, Y/Z) and/or Jacobian (X Z, Y Z^2, Z); infinity -> all zero
__global__ void k_msm_horner_finish(const fp *hom, g1_jac *out_jac, g1_aff *out_aff) {
    if (blockIdx.x != 0 || threadIdx.x != 0) return;
    fp X = hom[0], Y = hom[1], Z = hom[2];
    if (out_jac) {
        g1_jac j;
        if (fp_is_zero(Z)) pt_set_inf(j);
        else { fp z2; fp_mul_ni(j.x, X, Z); fp_sqr_ni(z2, Z); fp_mul_ni(j.y, Y, z2); j.z = Z; }
        *out_jac = j;
    }
    if (out_aff) {
        g1_aff a;
        fp zi;
        fp_inv_vartime(zi, Z);
        fp_mul_ni(a.x, X, zi);
        fp_mul_ni(a.y, Y, zi);
        *out_aff = a;
    }
}

// the G2 forms (window sums of the signature-side MSM; Jacobian result only)
__global__ void k_msm_horner_prep_g2(const g2_jac *W, size_t stride, int nwin, fp *hom) {
    const int w = blockIdx.x * blockDim.x + threadIdx.x;
    if (w >= nwin) return;
    g2_jac p = W[(size_t)w * stride];
    g2_jac_to_hom(hom + 6 * w, p);
}
__global__ void k_msm_horner_finish_g2(const fp *hom, g2_jac *out_jac, g2_aff *out_aff) {
    if (blockIdx.x != 0 || threadIdx.x != 0) return;
    fp2 X, Y, Z;
    X.c0 = hom[0]; X.c1 = hom[1]; Y.c0 = hom[2]; Y.c1 = hom[3]; Z.c0 = hom[4]; Z.c1 = hom[5];
    if (out_jac) {
        g2_jac j;
        if (fp2_is_zero(Z)) pt_set_inf(j);
        else { fp2 z2; fp2_mul(j.x, X, Z); fp2_sqr(z2, Z); fp2_mul(j.y, Y, z2); j.z = Z; }
        *out_jac = j;
    }
    if (out_aff) {
        g2_aff a;
        fp2 zi;
        fp2_inv_vartime(zi, Z);
        fp2_mul(a.x, X, zi);
        fp2_mul(a.y, Y, zi);
        *out_aff = a;
    }
}

// synthetic MSM inputs (benchmark only): P_i = [k_i]G1 with a 96-bit k_i, 255-bit coefficients
// (shape of benchmarks/bls12381_msm_g1.nim:22-44)
__global__ void BLS_LB k_msm_make_inputs(uint64_t seed, size_t n, g1_aff *points, uint8_t *scalars) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint64_t s = seed ^ (0xFACADEull + i * 0x100000001b3ull);
    uint64_t v[6];
    for (int k = 0; k < 6; k++) {
        s += 0x9e3779b97f4a7c15ull;
        uint64_t z = s;
        z = (z ^ (z >> 30)) * 0xbf58476d1ce4e5b9ull;
        z = (z ^ (z >> 27)) * 0x94d049bb133111ebull;
        v[k] = z ^ (z >> 31);
    }
    uint32_t kw[3] = {(uint32_t)v[0], (uint32_t)(v[0] >> 32), (uint32_t)v[1]};
    g1_jac g, r;
    g.x = G1_GEN_X; g.y = G1_GEN_Y; g.z = FP_ONE;
    pt_mul_words(r, g, kw, 3);
    g1_aff a;
    pt_to_affine(a, r);
    points[i] = a;
    for (int w = 0; w < 4; w++)
        for (int b = 0; b < 8; b++) scalars[32 * i + 8 * w + b] = (uint8_t)(v[2 + w] >> (8 * b));
    scalars[32 * i + 31] &= 0x7f;
}

// Stream-ordered: d_points (stride pstride bytes, aff_t<F> each) and d_scalars (stride sstride bytes, little-endian,
// nbits bits used) are device pointers; the sum lands in d_out_jac and/or d_out_aff (device, either may be null).
// p is the shape route::plan_msm chose for (n, nbits).  horner_prog, when set, launches the window-Horner dataflow
// program of that shape on (stream, homogeneous window sums, homogeneous result); otherwise k_msm_horner runs.
// No host synchronisation unless the scratch buffer has to grow.
template <class F>
static inline int msm_run(msm_state &st, const route::msm_plan &p,
                          const std::function<void(cudaStream_t, const fp *, fp *)> &horner_prog, const uint8_t *d_points,
                          size_t pstride, const uint8_t *d_scalars, size_t sstride, size_t n, int nbits, cudaStream_t s,
                          jac_t<F> *d_out_jac, aff_t<F> *d_out_aff, int *launches, std::string &err) {
    typedef jac_t<F> J;
    if (n >= ((size_t)1 << 31)) { err = "msm: too many points"; return -2; }
    const int sb = (nbits + 7) / 8;
    const int c = p.c, nwin = p.nwin, G = p.G;
    const size_t B = p.B, nseg = p.nseg;
    const size_t nb = (size_t)nwin * B, nsb = (nb + 1023) / 1024;
    const route::msm_layout o = route::msm_scratch(p, sizeof(J));
    cudaError_t e;
#define MCK(call) if ((e = (call)) != cudaSuccess) { err = std::string(#call ": ") + cudaGetErrorString(e); return -1; }
    if (st.bytes < o.total) {
        if (st.buf) { MCK(cudaStreamSynchronize(s)); if (st.tail) MCK(cudaStreamSynchronize(st.tail)); cudaFree(st.buf); }
        st.buf = nullptr;
        st.bytes = 0;
        MCK(cudaMalloc((void **)&st.buf, o.total));
        st.bytes = o.total;
    }
    if (G > 1 && !st.tail) {
        int lo_pri = 0, hi_pri = 0;
        MCK(cudaDeviceGetStreamPriorityRange(&lo_pri, &hi_pri));
        MCK(cudaStreamCreateWithPriority(&st.tail, cudaStreamNonBlocking, hi_pri));
        for (int i = 0; i < 8; i++) MCK(cudaEventCreateWithFlags(&st.ev_group[i], cudaEventDisableTiming));
        MCK(cudaEventCreateWithFlags(&st.ev_done, cudaEventDisableTiming));
        st.ev_ok = true;
    }
    uint32_t *counts = (uint32_t *)(st.buf + o.counts), *offsets = (uint32_t *)(st.buf + o.offsets);
    uint32_t *cursor = (uint32_t *)(st.buf + o.cursor), *rank = (uint32_t *)(st.buf + o.rank);
    uint32_t *bsums = (uint32_t *)(st.buf + o.bsums);
    uint32_t *biglist = (uint32_t *)(st.buf + o.big), *bigcount = (uint32_t *)(st.buf + o.bigcount);
    uint32_t *entries = (uint32_t *)(st.buf + o.entries);
    J *partials = (J *)(st.buf + o.partials), *buckets = (J *)(st.buf + o.buckets), *segs = (J *)(st.buf + o.segs);
    J *carry = (J *)(st.buf + o.carry);
    MCK(cudaMemsetAsync(counts, 0, nb * 4, s));
    MCK(cudaMemsetAsync(bigcount, 0, 4 * 8, s));
    int nl = 0;
    k_msm_count<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(d_scalars, sstride, n, sb, nbits, c, nwin, counts);
    k_msm_scan_blocks<<<(unsigned)nsb, 1024, 0, s>>>(counts, nb, bsums);
    k_msm_scan_top<<<1, 1024, 0, s>>>(bsums, nsb);
    k_msm_scan_apply<<<(unsigned)nsb, 1024, 0, s>>>(counts, nb, bsums, offsets, cursor, rank);
    k_msm_scatter<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(d_scalars, sstride, n, sb, nbits, c, nwin, cursor, entries);
    nl += 5;
    for (int g = 0; g < G; g++) {
        const int w0 = p.gw0[g + 1], wg = p.gw0[g] - p.gw0[g + 1];
        const size_t b0 = (size_t)w0 * B, b1 = b0 + (size_t)wg * B;
        const uint32_t K = p.K[g];
        const size_t gchunks = (n * (size_t)wg + K - 1) / K + 1;
        J *pg = partials + p.preg[g];
        k_msm_chunks<F><<<(unsigned)((gchunks + 127) / 128), 128, 0, s>>>(d_points, pstride, offsets, rank, entries, b0, b1, K, pg);
        cudaStream_t ts = s;
        if (G > 1) {
            MCK(cudaEventRecord(st.ev_group[g], s));
            MCK(cudaStreamWaitEvent(st.tail, st.ev_group[g], 0));
            ts = st.tail;
        }
        k_msm_combine<F><<<(unsigned)(((size_t)wg * B + 127) / 128), 128, 0, ts>>>(pg, offsets, rank, b0, b1, K, buckets, biglist, bigcount + g);
        k_msm_combine_big<F><<<128, 128, 0, ts>>>(pg, offsets, rank, b0, K, biglist, bigcount + g, buckets);
        size_t nt = (size_t)wg * nseg;
        J *sg = segs + (size_t)w0 * nseg;
        k_msm_segment<F><<<(unsigned)((nt + 127) / 128), 128, 0, ts>>>(buckets + b0, c, wg, (uint32_t)p.L, sg);
        nl += 4;
        for (size_t m = nseg; m > 1;) {
            size_t half = (m + 1) / 2;
            k_tree_rows<F><<<(unsigned)(((size_t)wg * half + 127) / 128), 128, 0, ts>>>(sg, wg, nseg, m, half);
            nl++;
            m = half;
        }
        if (p.horner_prog && horner_prog) {                  // p.horner_prog: G == 1
            constexpr bool is_g1 = std::is_same<F, fp>::value;
            constexpr int per = is_g1 ? 3 : 6;               // field elements per homogeneous point
            fp *hom = (fp *)(st.buf + o.hom);
            if constexpr (is_g1) k_msm_horner_prep<<<1, 128, 0, ts>>>(sg, nseg, nwin, hom);
            else k_msm_horner_prep_g2<<<1, 128, 0, ts>>>(sg, nseg, nwin, hom);
            horner_prog(ts, hom, hom + per * nwin);
            if constexpr (is_g1) k_msm_horner_finish<<<1, 32, 0, ts>>>(hom + per * nwin, d_out_jac, d_out_aff);
            else k_msm_horner_finish_g2<<<1, 32, 0, ts>>>(hom + per * nwin, d_out_jac, d_out_aff);
            nl += 2;                                         // horner_prog counts its own launch
        } else {
            k_msm_horner<F><<<1, 32, 0, ts>>>(sg, nseg, wg, c, g == 0, g == G - 1, carry, d_out_jac, d_out_aff);
            nl++;
        }
    }
    if (G > 1) {
        MCK(cudaEventRecord(st.ev_done, st.tail));
        MCK(cudaStreamWaitEvent(s, st.ev_done, 0));
    }
    MCK(cudaGetLastError());
#undef MCK
    if (launches) *launches += nl;
    return 0;
}

}  // namespace bls
