// route.hpp — the batch pipeline's route policy: which kernels a batch of n sets runs, and the measured size thresholds
// that decide it; the capacities of the Miller-loop workspaces, which every Miller plan must fit; and the shape of the
// Pippenger MSM (window width, segments, window groups, chunks, scratch layout).
// Plain C++ without CUDA, so that tests/hostsim compiles it and checks the plans on the host.
//
// Every threshold is read from the environment by read_thresholds() (INTEGRATION.md section 8); libblsgpu caches the
// result once per process.  The per-context switches (BLSGPU_SIDE_STREAM, BLSGPU_ACC_TEAM, BLSGPU_SERIAL_TAIL,
// BLSGPU_GRAPH) are read by blsgpu_create and come in through `switches`.  BLSGPU_PROG_FORMAT is the one variable read
// elsewhere, by fpprog.hpp, whose tests override it per thread.
#pragma once
#include <stddef.h>
#include <stdint.h>
#include <stdlib.h>

namespace route {

// Largest batches that take the warp-per-set programs: the cofactor / [r]sig programs (5-6 KB of shared memory per
// warp, 32 warps per SM) up to SMALL_MAX sets, the lines program (33 KB per warp, 6 per SM) up to SMALL_LINES_MAX
// pairs; beyond that a thread per set fills the machine better (tools/probe.py, profiles/).  SMALL_MAX is capped at the
// per-set stride of the small-route buffers.
static const size_t SMALL_ROUTE_CAP = 4096;
static const size_t SMALL_LINES_CAP = 16385;
static const unsigned ACC_BLOCK = 128;               // threads per block of k_miller_acc (BLS_ACC_BS)
static const unsigned LB_BLOCKS = 4;                 // resident 128-thread blocks per SM of the BLS_LB kernels (BLS_LB_BLOCKS)

enum { SMALL_HASH = 1, SMALL_SIG = 2, SMALL_LINES = 4, SMALL_GTPROD = 8 };   // bits of BLSGPU_SMALL_ROUTE

struct thresholds {
    size_t small_max, small_lines_max;
    int small_route;                                 // SMALL_* bits
    size_t pair_hash_min, pair_hash_max, pair_lines_max;
    size_t g2_msm_min, defer_sig_min;
    size_t g1_aside_max, g1_aside_large_min;
    size_t affine_block_min, h2d_slice_min;
    size_t chain_hog_min;
    int chain_wait;
    size_t graph_max, gt_prog_max, msm_after_hash_min;
    int map_lanes2, acc_old_rule;
    bool miller_g_set, miller_nseg_set;              // BLSGPU_MILLER_G / _NSEG override the shape rule of miller_shape
    int miller_g, miller_nseg;
    int msm_c, msm_l, msm_groups, msm_k;             // BLSGPU_MSM_C / _L / _GROUPS / _K override the MSM shape when > 0
    bool msm_horner_prog;                            // BLSGPU_MSM_HORNER_PROG=0 keeps the window Horner off the program
};

inline size_t env_size(const char *name, size_t def) { const char *e = getenv(name); return e ? (size_t)atoll(e) : def; }
inline int env_int(const char *name, int def) { const char *e = getenv(name); return e ? atoi(e) : def; }

inline thresholds read_thresholds() {
    thresholds t;
    t.small_max = env_size("BLSGPU_SMALL_MAX", 4096);
    if (t.small_max > SMALL_ROUTE_CAP) t.small_max = SMALL_ROUTE_CAP;
    t.small_lines_max = env_size("BLSGPU_SMALL_LINES_MAX", 1025);
    if (t.small_lines_max > SMALL_LINES_CAP) t.small_lines_max = SMALL_LINES_CAP;
    t.small_route = env_int("BLSGPU_SMALL_ROUTE", 15);
    // Two lanes per set for H(m_i) and the line evaluations (fp2h.cuh).  Introduced for mid-size batches, where a thread
    // per set leaves the machine under-filled; measured again at the end of round 2 (profiles/r2/r2_probe_routes_large.log)
    // it also wins for large ones: a block of lane pairs runs half as long as a block of threads, so the grid ends on a
    // finer wave boundary (81 920 sets: 43.1 -> 36.3 ms, 114 688: 52.6 -> 49.0), and the halved stacks stay in L2.
    // Lines: lane pairs up to 180 000 pairs; hash: up to 125 000 sets (at 131 072 the thread-per-set hash with its 1.73
    // waves is the quicker one: 55.0 ms against 55.4 with lane pairs for both and 55.8 with threads for both); beyond,
    // threads.
    t.pair_hash_min = env_size("BLSGPU_PAIR_HASH_MIN", 2049);
    t.pair_hash_max = env_size("BLSGPU_PAIR_HASH_MAX", 125000);
    t.pair_lines_max = env_size("BLSGPU_PAIR_LINES_MAX", 180000);
    // swept: 2 048 sets 6.54 -> 6.13 ms with the per-set programs, 2 600: 6.39 -> 6.33 with the MSM
    t.g2_msm_min = env_size("BLSGPU_G2_MSM_MIN", 2500);
    // Measured: 8 192 sets 8.10 -> 7.24 ms, 16 384: 11.1 -> 10.5, 32 768: 18.05 -> 17.2, 131 072: 57.7 -> 57.0; re-swept at
    // the end of the round: it pays from ~4 500 sets on (4 800: 7.0 -> 6.87 ms, 6 000: 7.2 -> 7.0; 4 096: 6.55 -> 6.60,
    // 3 000: 6.44 -> 6.51).
    t.defer_sig_min = env_size("BLSGPU_DEFER_SIG_MIN", 4500);
    // measured (profiles/r2): beside the hash up to 8 192 sets (4 096 sets: 7.4 -> 6.7 ms) and from 36 000 on (49 152:
    // 25.5 -> 24.1 ms, 65 536: 31.7 -> 30.3, 98 304: 45.8 -> 43.8, 131 072: 56.2 -> 55.9); between, the chain is short,
    // the two run side by side from the start and contend (9 000 sets: 8.4 -> 9.1 ms)
    t.g1_aside_max = env_size("BLSGPU_G1_ASIDE_MAX", 8192);
    t.g1_aside_large_min = env_size("BLSGPU_G1_ASIDE_LARGE_MIN", 36000);
    t.affine_block_min = env_size("BLSGPU_AFFINE_BLOCK_MIN", 1025);
    t.h2d_slice_min = env_size("BLSGPU_H2D_SLICE_MIN", 32768);
    t.chain_hog_min = env_size("BLSGPU_CHAIN_HOG_MIN", 1024);
    t.chain_wait = env_int("BLSGPU_CHAIN_WAIT", 1);
    t.graph_max = env_size("BLSGPU_GRAPH_MAX", 8192);
    t.gt_prog_max = env_size("BLSGPU_GT_PROG_MAX", (size_t)1 << 20);
    // Off by default: the signature-side MSM waits for the hash kernel and runs beside [r_i]pk_i and the line evaluations
    // instead.  Measured at 131 072 sets: hash 26.1 -> 24.0 ms (its time alone), [r_i]pk_i +0.9, lines +1.3, step 57.3 ->
    // 57.1 ms whatever the length of the scalar chain — but the starved MSM then ends only 1-2 ms before the join, so the
    // gain is not worth the exposure.
    t.msm_after_hash_min = env_size("BLSGPU_MSM_AFTER_HASH_MIN", ~(size_t)0);
    t.map_lanes2 = env_int("BLSGPU_MAP_LANES2", 1);
    t.acc_old_rule = env_int("BLSGPU_ACC_OLD_RULE", 0);
    const char *g = getenv("BLSGPU_MILLER_G"), *ns = getenv("BLSGPU_MILLER_NSEG");
    t.miller_g_set = g != nullptr;
    t.miller_g = g ? atoi(g) : 0;
    t.miller_nseg_set = ns != nullptr;
    t.miller_nseg = ns ? atoi(ns) : 0;
    t.msm_c = env_int("BLSGPU_MSM_C", 0);
    t.msm_l = env_int("BLSGPU_MSM_L", 0);
    t.msm_groups = env_int("BLSGPU_MSM_GROUPS", 0);
    t.msm_k = env_int("BLSGPU_MSM_K", 0);
    t.msm_horner_prog = env_int("BLSGPU_MSM_HORNER_PROG", 1) != 0;
    return t;
}

struct switches { bool use_side, acc_team, serial_tail, use_graph; };

// the RLC scalar chains of a batch of total_n sets derived in `chunks` reference chunks: one per chunk
inline size_t rlc_chains(size_t total_n, uint32_t chunks) {
    return chunks == 0 ? 1 : (total_n < chunks ? total_n : (size_t)chunks);
}

// Long chains (thousands of sequential SHA-256 blocks per reference chunk) are pure single-warp latency, and every
// consumer of the scalars waits for them.  Sharing an SM with the hash kernel's 16 warps costs the chain warp half of
// its issue slots (measured: 24-31 ms instead of 13 ms for 8 192 blocks per chain), so from CHAIN_HOG_MIN blocks per
// chain on a block of chains asks for the whole shared memory of an SM and therefore gets one to itself: 32 chains per
// block, one SM per 32 chunks.
inline bool chain_hog(const thresholds &t, size_t total_n, uint32_t chunks) {
    return total_n / rlc_chains(total_n, chunks) >= t.chain_hog_min;
}

// H(m_i) as per-set programs: bit 0 of SMALL_ROUTE, up to SMALL_MAX sets.  Aggregate verification applies this rule
// alone; a batch leaves the sizes of the lane-pair hash to it.
inline bool program_hash(const thresholds &t, size_t n, bool serial_tail) {
    return (t.small_route & SMALL_HASH) && n <= t.small_max && !serial_tail;
}

// H(m_i): map + cofactor program / k_hash_sets_lanes2 / k_hash_sets_pair / k_hash_sets
enum { HASH_PROGRAM, HASH_LANES2, HASH_PAIR, HASH_THREAD };
// sum_i [r_i] sig_i: per-set program or k_g2_mul, each followed by a tree / Pippenger
enum { SIG_PROGRAM, SIG_MUL, SIG_MSM };
// k_pairs_affine: AFF_B sets per thread / a warp per set / one inversion per block
enum { AFFINE_DEFAULT, AFFINE_WARP, AFFINE_BLOCK };

struct batch_plan {
    int hash;              // HASH_*
    bool sliced;           // the host copy is cut into pieces, each hashed on its own stream as it lands
    bool small;            // small-route buffers and per-set programs (cofactor, [r_i] sig_i)
    int sig;               // SIG_*
    bool g1_aside;         // [r_i] pk_i on the third stream, beside the hash
    bool msm_after_hash;   // the signature-side MSM waits for the hash kernel
    bool defer_sig;        // the pair (S, -G1) gets its own one-pair Miller loop on the side stream
    int affine;            // AFFINE_*
    bool chain_hog;        // the scalar chains reserve whole SMs
    bool chain_wait;       // the main stream waits until the chains' block is placed
    bool graph;            // replayed from a captured CUDA graph (the caller also needs the random bytes)
    bool copy_ahead;       // blsgpu_batch_verify copies a host batch of this size before the pipeline, so that a graph
                           // captured for it starts from the device copy; larger ones are copied by the pipeline itself
};

// n sets of a batch of total_n; host_src: the pipeline copies the sets from the caller's host buffer itself
inline batch_plan plan_batch(const thresholds &t, const switches &sw, size_t n, size_t total_n, uint32_t chunks, bool host_src,
                             bool scalars) {
    batch_plan p;
    p.sliced = host_src && n >= t.h2d_slice_min && n > t.small_max;
    p.small = t.small_route != 0 && n <= t.small_max && !sw.serial_tail;
    const bool pair_hash = n >= t.pair_hash_min && n <= t.pair_hash_max;
    if (p.sliced) p.hash = pair_hash ? HASH_LANES2 : HASH_THREAD;
    else if (program_hash(t, n, sw.serial_tail) && !pair_hash) p.hash = HASH_PROGRAM;
    else if (pair_hash) p.hash = HASH_LANES2;
    else if (n <= 8192) p.hash = HASH_PAIR;
    else p.hash = HASH_THREAD;
    // Pippenger over the signatures in place for batches that can fill the buckets, n independent 64-bit
    // multiplications + tree below that
    if (n >= t.g2_msm_min) p.sig = SIG_MSM;
    else p.sig = p.small && (t.small_route & SMALL_SIG) ? SIG_PROGRAM : SIG_MUL;
    // Small batches are latency chains (one thread per set): [r_i]pk_i does not depend on H(m_i), so it leads the
    // third stream instead of queueing behind the hash kernel.  Large batches: behind a scalar chain of several
    // milliseconds it starts while the hash kernel is in its last wave and fills the slots that wave leaves empty.
    p.g1_aside = sw.use_side && (n <= t.g1_aside_max || n >= t.g1_aside_large_min);
    p.msm_after_hash = sw.use_side && n >= t.msm_after_hash_min;
    // the n set pairs do not wait for the signature sum (scalar chain, then the signature-side MSM: 4 ms at 8 192 sets,
    // tens of milliseconds behind the long chains of a large batch)
    p.defer_sig = sw.use_side && !sw.serial_tail && n >= t.defer_sig_min && !scalars;
    // small batches: one inversion per set is pure latency -> binary Euclid, one working lane per warp (it diverges
    // across the lanes of a warp: sharing warps it is no quicker than the uniform Fermat chain, 0.53 vs 0.46 ms at 129)
    p.affine = n >= t.affine_block_min ? AFFINE_BLOCK : (p.small ? AFFINE_WARP : AFFINE_DEFAULT);
    p.chain_hog = !scalars && chain_hog(t, total_n, chunks);
    p.chain_wait = t.chain_wait && p.chain_hog && sw.use_side;
    p.graph = sw.use_graph && !scalars && n <= t.graph_max && !sw.serial_tail;
    p.copy_ahead = host_src && n <= t.graph_max;
    return p;
}

// Work decomposition of the accumulation: G pairs per group (they share the Fp12 squarings) and nseg loop segments,
// chosen so that groups x segments gives every SM several warps even for small batches.
inline void miller_shape(const thresholds &t, size_t np, bool team, int &G, int &nseg) {
    if (team && np <= 8192) {
        // Latency regime (the machine is not full).  Measured on B200 (tools/gpu_small_sweep.sh): a team spends ~7.5 us
        // per (squaring or line) step while all teams are resident (~12k of them), the product over groups is one
        // block-wide tree (0.59 ms) up to 128 groups and two launches (1.16 ms) beyond (0.084 ms per tree level); up to 64 groups it is a pair of product-tree programs,
        // one warp per row (0.04-0.08 ms), the segment Horner program costs
        // 0.22 ms + 7.4 us per segment.
        double best = 0.0;
        G = 1; nseg = 32;
        for (int g = 1; g <= 64; g *= 2)
            for (int ns = 4; ns <= 32; ns *= 2) {
                const size_t ngroups = (np + g - 1) / g;
                if (ngroups * ns > 32768) continue;             // d_F holds at least 40 000 (group, segment) products
                const double waves = (double)((ngroups * ns + 11999) / 12000);
                const double acc = waves * (double)((63 + ns - 1) / ns) * (1 + g) * (g <= 16 ? 7.5e-3 : 9.5e-3);
                int levels = 0;                                 // product trees of eight (k_fp_program_rows), ~0.03 ms a level
                for (size_t m = ngroups; m > 1; m = (m + 7) / 8) levels++;
                int depth = 0;
                while (((size_t)1 << depth) < ngroups) depth++;
                const double gtp = t.acc_old_rule ? (ngroups <= 8 ? 0.04 : (ngroups <= 64 ? 0.08 : (ngroups <= 128 ? 0.084 * depth : 1.16)))
                                           : 0.01 + 0.03 * levels;
                const double cost = acc + gtp + 0.22 + 7.4e-3 * ns;
                if (best == 0.0 || cost < best) { best = cost; G = g; nseg = ns; }
            }
    } else if (team) {
        // Throughput regime.  The Fp12 squarings of a step are shared by the G pairs of a group (work per pair ~ 884 + 756 / G
        // multiplications), and short segments keep the tail of the grid short: swept on B200 (profiles/r2): 16 384 sets
        // G = 8 / 16 segments (2.14 -> 1.82 ms), 32 768 and 65 536: G = 16 / 16 (3.79 -> 3.51, 7.08 -> 6.59), 131 072:
        // G = 24 / 8 (14.3 -> 13.1 ms); past ~65 000 teams the product trees and the segment Horner eat the gain.
        if (t.acc_old_rule) {
            G = 1;
            while (G < 16 && np / (size_t)(2 * G) >= 4096) G *= 2;
            size_t ngroups = (np + G - 1) / G;
            size_t want = ((size_t)1 << 15) / ngroups;
            nseg = want < 1 ? 1 : (want > 32 ? 32 : (int)want);
        } else {
            G = np < 24576 ? 8 : (np < 98304 ? 16 : 24);
            const size_t ngroups = (np + G - 1) / G;
            nseg = 16;
            while (nseg > 4 && ngroups * (size_t)nseg > 65536) nseg -= 4;
        }
    } else {
        G = 1;
        while (G < 8 && np / (size_t)(2 * G) >= 8192) G *= 2;
        size_t ngroups = (np + G - 1) / G;
        size_t want = ((size_t)1 << 17) / ngroups;
        nseg = want < 1 ? 1 : (want > 32 ? 32 : (int)want);
    }
    if (t.miller_g_set) G = t.miller_g;
    if (t.miller_nseg_set) nseg = t.miller_nseg;
    if (G < 1) G = 1;
    if (nseg < 1) nseg = 1;
    if (nseg > 63) nseg = 63;
}

enum { LINES_PROGRAM, LINES_LANES2, LINES_THREAD };   // per-pair program + scatter / k_miller_lines_lanes2 / k_miller_lines

// Miller-loop tiling: at most LINES_TILE pairs have their 68 x 288-byte line triples resident at once
static const size_t LINES_TILE = (size_t)1 << 18;

// Capacities of a Miller-loop workspace (blsgpu.cu miller_ws)
struct miller_caps {
    size_t lines_cap;      // pairs per tile of the lines buffer
    size_t f_cap;          // entries of the block products F
    size_t f2_cap;         // entries of the second-level block products F2
    size_t small_lines;    // pairs of the lines-program buffer (allocated on first use)
};

// the workspace of the batch's Miller loop in a context of max_sets sets: the set pairs + the signature-side pair
// (tests/test_hostsim.py checks that the plans of 1 to max_sets + 1 pairs fit it)
inline miller_caps miller_caps_batch(const thresholds &t, size_t max_sets) {
    const size_t n = max_sets;
    miller_caps c;
    c.lines_cap = ((n + 1 < LINES_TILE ? n + 1 : LINES_TILE) + 31) & ~(size_t)31;
    // block products: <= 64 segments x (blocks per tile + 1) x tiles
    c.f_cap = (n + 1) / 2 + 40000 + 64 * ((n + 1) / LINES_TILE + 2);   // >= nseg * groups for every miller_shape
    c.f2_cap = c.f_cap / 8 + 4096;                          // level-1 output of the 8-way product trees (+ padding)
    c.small_lines = t.small_lines_max;
    return c;
}

// the workspace of the deferred signature pair's one-pair Miller loop
inline miller_caps miller_caps_sig() { return {32, 2048, 512, 2}; }

struct miller_plan {
    int G, nseg;
    int lines;             // LINES_* of every tile of lines_cap pairs but the last
    int lines_last;        // LINES_* of the last tile (the only one when np <= lines_cap)
    size_t ncols;          // entries per segment row of the block products
    bool gt_prog;          // the GT product of each segment row runs as product-tree programs over groups of 8 columns
    size_t row_stride;     // entries between segment rows of F
    size_t ncols2;         // entries per segment row of F2
};

// np pairs, tiled by lines_cap (the pairs whose line triples fit the workspace at once)
inline miller_plan plan_miller(const thresholds &t, size_t np, size_t lines_cap, bool team, bool serial_tail) {
    miller_plan p;
    miller_shape(t, np < lines_cap ? np : lines_cap, team, p.G, p.nseg);
    p.ncols = 0;
    for (size_t off = 0; off < np; off += lines_cap) {
        const size_t tile = np - off < lines_cap ? np - off : lines_cap;
        const size_t ngroups = (tile + p.G - 1) / p.G;
        p.ncols += team ? ngroups : (ngroups + ACC_BLOCK - 1) / ACC_BLOCK;
    }
    const bool single = np <= lines_cap;
    p.gt_prog = (t.small_route & SMALL_GTPROD) && team && single && p.ncols <= t.gt_prog_max && !serial_tail;
    // small batches: the GT product of each segment row runs as product-tree programs over groups of 8 columns, so
    // the rows of F are padded to a multiple of 8 with ones
    p.row_stride = p.gt_prog && p.ncols > 8 ? ((p.ncols + 7) & ~(size_t)7) : p.ncols;
    p.ncols2 = p.gt_prog ? ((((p.ncols + 7) / 8) + 7) & ~(size_t)7) : (p.ncols + ACC_BLOCK - 1) / ACC_BLOCK;
    // one warp per pair runs the 68 line evaluations as a dataflow program (two multiplication levels per tangent
    // instead of ~20 dependent products)
    if ((t.small_route & SMALL_LINES) && single && np <= t.small_lines_max && !serial_tail) {
        p.lines = p.lines_last = LINES_PROGRAM;
    } else {
        const size_t last = np - (np - 1) / lines_cap * lines_cap;
        p.lines = (single ? np : lines_cap) <= t.pair_lines_max ? LINES_LANES2 : LINES_THREAD;
        p.lines_last = last <= t.pair_lines_max ? LINES_LANES2 : LINES_THREAD;
    }
    return p;
}

// the plan's block products fit the workspace
inline bool fits(const miller_plan &p, const miller_caps &c) {
    return (size_t)p.nseg * p.row_stride <= c.f_cap && (size_t)p.nseg * p.ncols2 <= c.f2_cap;
}

// Window width c and count.  Cost model per candidate c: nwin * (11 n + 32 * 2^(c-1)) field multiplications (one
// mixed addition per non-zero digit, two full additions per bucket in the reduction).  Signed digits put bit `nbits`
// (the last carry) into the top window; a top window of only a few bits would funnel n / 2^bits entries into each of
// its few buckets, so widths that leave it fewer than 6 bits are skipped (for nbits = 255: c = 16, 13, 10, 8 qualify).
inline void msm_shape(const thresholds &t, size_t n, int nbits, int &c, int &nwin) {
    int lg = 0;
    while ((n >> (lg + 1)) != 0) lg++;
    int best_c = 0;
    double best = 0.0;
    const int hi = lg - 2 > 16 ? 16 : lg - 2, lo = lg - 8 < 2 ? 2 : lg - 8;
    for (int cc = hi; cc >= lo; cc--) {
        const int nw = (nbits + 1 + cc - 1) / cc, top = nbits + 1 - (nw - 1) * cc;
        if (nw > 1 && top < (cc < 6 ? cc : 6)) continue;
        const double cost = (double)nw * (11.0 * (double)n + 32.0 * (double)((size_t)1 << (cc - 1)));
        if (!best_c || cost < best) { best_c = cc; best = cost; }
    }
    if (!best_c) best_c = lg - 4 < 2 ? 2 : (lg - 4 > 16 ? 16 : lg - 4);
    c = t.msm_c > 0 ? t.msm_c : best_c;
    nwin = (nbits + 1 + c - 1) / c;
}

struct msm_plan {
    int c, nwin;           // window width, windows
    size_t B;              // buckets per window: digit magnitudes 1 .. 2^(c-1)
    size_t L, nseg;        // buckets per segment, segments per window
    int G;                 // window groups, top windows first
    int gw0[9];            // group g = windows [gw0[g+1], gw0[g]) counted from the top
    uint32_t K[8];         // entries per chunk of group g
    size_t preg[9];        // partial-slot region of group g: [preg[g], preg[g+1])
    size_t emax;           // entries of the bucket-sorted list: n * nwin
    bool horner_prog;      // the window Horner may run as a dataflow program (if its program builds)
};

// n points with nbits-bit scalars on a device of `sms` SMs
inline msm_plan plan_msm(const thresholds &t, size_t n, int nbits, int sms) {
    msm_plan p;
    msm_shape(t, n, nbits, p.c, p.nwin);
    p.B = (size_t)1 << (p.c - 1);
    p.emax = n * (size_t)p.nwin;
    const size_t wave = (size_t)sms * LB_BLOCKS * 128;
    size_t L = p.B / 512;                          // segment length: short serial chains, <= 512 segments per window
    if (L < 4) L = 4;
    if (L > 32) L = 32;
    if (t.msm_l > 0) L = (size_t)t.msm_l;
    if (L > p.B) L = p.B;
    p.L = L;
    p.nseg = p.B / L;
    // Window groups, top windows first.  The tail of a group is latency-bound (a few thousand threads, then one), so
    // it runs on the tail stream while the main stream accumulates the buckets of the next group.
    int G = t.msm_groups > 0 ? t.msm_groups : 1;
    if (G > 8) G = 8;
    if (G > p.nwin) G = p.nwin;
    p.G = G;
    p.gw0[0] = p.nwin;
    for (int g = 0; g < G; g++) p.gw0[g + 1] = p.nwin - (int)(((size_t)p.nwin * (g + 1)) / G);
    // entries per chunk, per group: the chunk grid of a group fills whole waves of the resident-thread capacity
    // (SMs x 4 blocks x 128) with about 32 additions per thread; short MSMs get one wave of shorter chunks
    p.preg[0] = 0;                                 // partial slots of a group: its chunks + its buckets + 1
    for (int g = 0; g < G; g++) {
        const size_t wg = (size_t)(p.gw0[g] - p.gw0[g + 1]), eg = n * wg;
        size_t waves = eg / (wave * 32);
        if (waves < 1) waves = 1;
        size_t Kz = (eg + waves * wave - 1) / (waves * wave);
        if (Kz < 8) Kz = 8;
        if (t.msm_k > 0) Kz = (size_t)t.msm_k;
        p.K[g] = (uint32_t)Kz;
        p.preg[g + 1] = p.preg[g] + (eg + Kz - 1) / Kz + 1 + wg * p.B + 1;
    }
    p.horner_prog = G == 1 && p.nwin <= 128 && t.msm_horner_prog;
    return p;
}

// byte offsets into the MSM's scratch buffer, for Jacobian points of jac_bytes bytes
struct msm_layout { size_t counts, offsets, cursor, rank, bsums, big, bigcount, carry, hom, entries, partials, buckets, segs, total; };

inline msm_layout msm_scratch(const msm_plan &p, size_t jac_bytes) {
    const size_t nb = (size_t)p.nwin * p.B, nsb = (nb + 1023) / 1024;   // buckets, scan blocks
    auto al = [](size_t x) { return (x + 255) & ~(size_t)255; };
    msm_layout o;
    o.counts = 0;
    o.offsets = o.counts + al(nb * 4);
    o.cursor = o.offsets + al((nb + 1) * 4);
    o.rank = o.cursor + al(nb * 4);
    o.bsums = o.rank + al((nb + 1) * 4);
    o.big = o.bsums + al(nsb * 8);
    o.bigcount = o.big + al(nb * 4);
    o.carry = o.bigcount + 256;
    o.hom = o.carry + al(jac_bytes);
    o.entries = o.hom + al((size_t)(6 * p.nwin + 6) * 48);
    o.partials = o.entries + al(p.emax * 4);
    o.buckets = o.partials + al(p.preg[p.G] * jac_bytes);
    o.segs = o.buckets + al(nb * jac_bytes);
    o.total = o.segs + al((size_t)p.nwin * p.nseg * jac_bytes);
    return o;
}

}  // namespace route
