// simplex_cta.cuh — one-CTA-per-LP dense two-phase revised simplex (the "wave" kernel).
//
// Replaces, for a whole batch / frontier wave at once, the reference's per-node call chain
//   subProblem.solve            /root/reference/subproblem.go:141-187
//     combineInequalities       subproblem.go:55-78      (branch rows synthesised on the fly, never stored)
//     convertToEqualities       subproblem.go:81-139     ([A0 0; G I] read through src_a(), never materialised)
//     lp.Simplex                vendor/gonum.org/v1/gonum/optimize/convex/lp/simplex.go:88-302
//       verifyInputs :385-439, findInitialBasic :492-607, findLinearlyIndependent :611-637,
//       computeMove :306-342, replaceBland :347-383, initializeFromBasic :447-471
// The DECISIONS are Gonum's: Dantzig pricing with floats.MinIdx first-position ties over the
// positional non-basic list that is mutated by swaps (simplex.go:174-184,280), ratio test by MinIdx
// over positions, Bland fallback when the step is <= 0, every tolerance of simplex.go:42-58, Phase I
// with one artificial column and tol 1e-10, the artificial-still-basic repair scan.
// The ARITHMETIC is not Gonum's: instead of three fresh LU factorisations per pivot the basis inverse
// is kept explicitly (m x m, row-major) and updated by a rank-1 (product-form) step; it is rebuilt by
// Gauss-Jordan inversion with partial pivoting every `refactor_period` pivots and once more before an
// optimal basis is reported ("polish"), so the returned x comes from fresh factors like Gonum's.
//
// Data layout per LP (shared memory when it fits, else a per-CTA slice of an HBM workspace):
//   W   m x ldw   working copy of [A | artificial] with COLUMNS PERMUTED: columns 0..m-1 are the basic
//                 columns in basis-position order, columns m.. are the non-basic ones in list-position
//                 order; a pivot swaps two columns. Row-major with odd ldw: pricing (thread per
//                 column) and column extraction (thread per row) are both bank-conflict free.
//   Bi  m x ldb   basis inverse, row-major, odd ldb.
//   vectors       xb, cb, y (duals), al (B^-1 a_e), mv (ratios), bv (rhs), prow, art, t1, t2, cn, r.
// Tier 1 (SolverT<true>) differs: Bi lives in registers and W keeps the ORIGINAL column order (column v of
// W is column v of A, column n the artificial); the positional lists basic[] / nonbasic[] are the only
// thing a pivot permutes, so no column ever moves.
// All reductions that pick an index return the FIRST minimum (value, position) like floats.MinIdx.
#pragma once
#include <math.h>
#include <limits.h>

#include "../../include/gomilp_status.h"
#include "cta_rt.cuh"

namespace gm {

struct BatchParams {
    // ---- problem source (device pointers) -------------------------------------------------------
    const double* c;  // [count][n0] or one shared root
    const double* A;  // [count][m0][lda] row-major (Gonum mat.Dense layout) or one shared root
    const double* b;  // [count][m0]
    long long c_stride, A_stride, b_stride;  // doubles between consecutive LPs; 0 = shared root
    int lda;
    int m0, n0;  // root shape
    int L;       // branch rows appended per node (wave mode); 0 for plain batches
    const int* bvar;      // [count][L] variable of each bnbConstraint (subproblem.go:36-44)
    const double* bsign;  // [count][L] gsharp[var] = +1 / -1
    const double* brhs;   // [count][L] hsharp
    const long long* initial_basic;  // [count][m] or nullptr (simplex.go:147-160)
    // Warm start of B&B children (north star "children warm-start from the parent basis"): node k continues from
    // node warm_parent[k] of the PREVIOUS wave (depth L-1), whose final basis / inverse are kept in HBM.
    const int* warm_parent;          // [count] index into the previous wave, -1 = cold start; nullptr = all cold
    const long long* warm_basis;     // [prev_count][m-1]
    const double* warm_bi;           // [prev_count][(m-1)*(m-1)] row-major basis inverses of the previous wave
    double* bi_out;                  // [count][m*m] or nullptr: final basis inverse of every node (for the next wave)
    double tol;
    int count;
    int max_pivots;       // safety cap (the reference has none); <=0: 50*(m+n)+1000
    int refactor_period;  // pivots between Gauss-Jordan rebuilds of Bi; <=0: 100 (HBM tiers: max(100, 2m))
    int ring_stages, ring_stage_bytes;  // HBM tier: TMA staging ring in shared memory (0: none)
    int stream_min_m;                   // rows shorter than this use plain loads (bulk copies pay off for long rows)
    int tier;             // 1..5, see gm_timing.tier (selects where the generic kernel finds W / Bi / vectors)
    int hbm_layout;       // 1: W / Bi live in HBM (row strides padded to 32 B instead of to an odd count)
    // ---- outputs --------------------------------------------------------------------------------
    int* status;        // [count] gm_status
    double* optF;       // [count]
    double* x;          // [count][x_stride], first x_len entries written (n, or n0 in wave mode)
    long long x_stride;
    int x_len;
    long long* basis;  // [count][m] or nullptr; -1 when the reference returns nil
    int* stats;        // [count][8] or nullptr: pivots phase I, phase II, bland calls, inversions,
                       //   used phase I, basis-scan fallback used, repair trials, x non-nil
    // ---- work -----------------------------------------------------------------------------------
    double* work;           // HBM workspace for the tiers that need one: [gridDim][work_stride]
    long long work_stride;  // doubles per CTA
    int* queue;             // work-queue counter (zeroed before launch)
    int robust;             // non-reference: an LP on which the reference's rule set gives up (Bland dead end, numerically
                            // singular basis after zero-step pivots, cycling) is re-solved on a slightly perturbed rhs
    const int* ready;       // optional: number of LPs whose inputs have ARRIVED in HBM (written by the copy stream while
                            // the kernel runs, see engine.cu run_host_batch_streamed); nullptr = everything is resident
    const int* lp_list;     // optional: work item k solves LP lp_list[k] (retry launches); nullptr = identity
    // ---- pivot trace (parity evidence): LP `trace_lp` records (phase, entering variable, leaving variable, bland)
    // for its first `trace_cap` pivots. Only the WARM-capable kernels carry the code (the bench kernel does not).
    int* trace;
    int trace_cap, trace_lp;
    // ---- cooperative tier (6): `coop_G` CTAs of one cooperative launch work on one LP (simplex_wave_coop) --------
    int coop_G;                     // CTAs per group
    int coop_pan;                   // inversion panel width when the panel fits in shared memory (16), else 0
    int coop_small;                 // 1: groups of one CTA keep the solver's vectors in shared memory (see CoopLayout)
    unsigned long long* coop_bar;   // [groups] barrier counters, zeroed before launch
    long long* prof;                // optional [count][8]: leader clock cycles spent per activity (see coop_cta_main)
};

// Workspace of one CTA, split in a "big" part (W and Bi: O(mn) doubles) and a "small" part (vectors,
// index lists, reduction scratch: O(m+n)). Tier 1 keeps both in shared memory, tier 2 keeps the big
// part in HBM and the small part in shared memory, tier 3 keeps both in HBM.
struct WsLayout {
    int ldw, ldb, nn1, wrows, vlen;
    size_t W, Bi;         // offsets in doubles inside the big part
    size_t big_doubles;
    size_t xb, cb, y, al, mv, bv, prow, art, t1, t2, cn, r, red;  // offsets in doubles inside the small part
    size_t small_doubles;
    size_t basic, nonbasic, inb, redi, ipiv, cperm;  // offsets in ints, after the small doubles
    size_t n_ints;
    size_t big_bytes, small_bytes;
};

// reg = the register-resident tier (m <= 64, 256 threads): Bi lives in registers, the "Bi" slot of the
// workspace becomes a 64 x 68 staging tile, W gets a row stride = 4 (mod 16) and rows padded to a
// multiple of 4, and every m-vector is padded to 64 entries (see SolverT<true>).
#ifdef __CUDACC__
__host__ __device__
#endif
inline WsLayout ws_layout(int m, int n, int T, bool reg = false, bool hbm = false, bool bi_smem = false) {
    WsLayout w;
    if (reg) {
        int ld = n + 1;
        while ((ld & 15) != 4) ++ld;
        w.ldw = ld;
        w.ldb = 68;
        w.wrows = 64;
        w.vlen = 64;
    } else {
        w.ldw = hbm ? ((n + 2 + 3) & ~3) : ((n + 1) | 1);
        w.ldb = hbm ? ((m + 3) & ~3) : (m | 1);
        if (bi_smem) {  // quad-mapped loop: 8 rows x 4 consecutive columns per warp access -> stride = 4 (mod 16)
            int ld = m;
            while ((ld & 15) != 4) ++ld;
            w.ldb = ld;
        }
        w.wrows = m;
        w.vlen = m;
    }
    w.nn1 = (n + 1 - m) > 1 ? (n + 1 - m) : 1;
    size_t o = 0;
    w.W = o; o += (size_t)w.wrows * w.ldw;
    w.Bi = o; o += reg ? (size_t)64 * 68 : (size_t)m * w.ldb;
    w.big_doubles = o;
    o = 0;
    const size_t v = (size_t)w.vlen;
    w.xb = o; o += v;
    w.cb = o; o += v;
    w.y = o; o += v;
    w.al = o; o += v;
    w.mv = o; o += v;
    w.bv = o; o += v;
    w.prow = o; o += v;
    w.art = o; o += v;
    w.t1 = o; o += v;
    w.t2 = o; o += v;
    w.cn = o; o += w.nn1;
    w.r = o; o += w.nn1;
    w.red = o; o += T;
    w.small_doubles = o;
    size_t q = 0;
    w.basic = q; q += m;
    w.nonbasic = q; q += w.nn1;
    w.inb = q; q += n + 1;
    w.redi = q; q += T;
    w.ipiv = q; q += m;
    w.cperm = q; q += 64;
    w.n_ints = q;
    w.big_bytes = w.big_doubles * sizeof(double);
    w.small_bytes = w.small_doubles * sizeof(double) + ((w.n_ints * sizeof(int) + 7) / 8) * 8;
    return w;
}

struct MinLoc {
    double v;
    int i;
};

// Cooperative tier: what one group of G CTAs keeps in HBM after the generic workspace (ws_layout with hbm = true),
// and what each of its CTAs keeps in shared memory. Offsets in doubles.
struct CoopLayout {
    size_t Bi1, Tp, Rs, mail, group_doubles;              // HBM, relative to the group's slice
    size_t s_y, s_prow, s_ae, s_xb, s_al, s_f, s_r, s_part, s_red, s_bit, s_redi, smem_bytes;  // shared memory
    int pan_nb;  // 16: the inversion panel lives in shared memory (aliasing the main-loop scratch); 0: in HBM, 32 wide
    size_t s_small;     // G == 1 only: the solver's vectors / index lists live in shared memory too (nobody else reads
    int small_in_smem;  // them), which is what makes the leader's serial phases cheap on wide waves of mid-size LPs
};
#ifdef __CUDACC__
__host__ __device__
#endif
inline CoopLayout coop_layout(int m, int n, int T, int G, size_t smem_limit = 200 * 1024) {
    const WsLayout w = ws_layout(m, n, T, false, true);
    CoopLayout c;
    auto up4 = [](size_t v) { return (v + 3) & ~(size_t)3; };
    size_t o = up4(w.big_doubles + w.small_bytes / 8 + 8);
    c.Bi1 = o; o = up4(o + (size_t)m * w.ldb);
    c.Tp = o; o = up4(o + (size_t)m * 32);
    c.Rs = o; o = up4(o + (size_t)32 * w.ldb);
    c.mail = o; o = up4(o + 16 + 12 * (size_t)G);
    c.group_doubles = o;
    const size_t mp = (size_t)((m + 3) & ~3);
    const size_t rlen = (size_t)(((n + 1 - m) > m ? (n + 1 - m) : m) + 4) & ~(size_t)3;
    size_t q = 0;
    c.s_y = q; q += mp;
    c.s_prow = q; q += mp;
    c.s_ae = q; q += mp;
    c.s_xb = q; q += mp;
    c.s_al = q; q += mp;
    c.s_f = q; q += mp;
    c.s_r = q; q += rlen;
    c.s_part = q; q += (size_t)T + mp;
    // The inversion panel (m x 17 doubles, 16 columns + 1 of padding) plus a column and a row vector ALIAS the
    // main-loop scratch above: an inversion only runs between main-loop calls, when all of it is dead.
    const size_t pan = (size_t)m * 17 + mp + 32;
    const size_t tail = 2 * (size_t)T + (mp + 1) / 2 + (2 * (size_t)T + 1) / 2;
    c.pan_nb = ((pan > q ? pan : q) + tail) * sizeof(double) + 1024 <= smem_limit ? 16 : 0;
    if (c.pan_nb && pan > q) q = pan;
    c.s_red = q; q += 2 * (size_t)T;    // two halves, used alternately by the block reductions
    c.s_bit = q; q += (mp + 1) / 2;     // ints
    c.s_redi = q; q += (2 * (size_t)T + 1) / 2;  // ints
    q = (q + 1) & ~(size_t)1;
    c.s_small = q;
    c.small_in_smem = (G == 1 && (q * sizeof(double) + w.small_bytes + 1024 <= smem_limit)) ? 1 : 0;
    if (c.small_in_smem) q += w.small_bytes / sizeof(double) + 2;
    c.smem_bytes = q * sizeof(double);
    return c;
}

// WARM = compiled with the warm-start entry / basis-inverse output paths (gm_solve_wave_warm); the cold
// instantiation of the register tier is kept free of them because they cost registers in the hot loop.
template <bool REG, bool WARM = true, bool COOP = false>
struct SolverT {
    // problem
    int m, n, m0, n0, L, lda;
    const double *c0, *A0, *b0;
    const int* bvar;
    const double *bsign, *brhs;
    // workspace
    double *W, *Bi, *xb, *cb, *y, *al, *mv, *bv, *prow, *art, *t1, *t2, *cn, *r, *red;
    int *basic, *nonbasic, *inb, *redi, *ipiv, *cperm;
    int ldw, ldb;
    // REG tier: thread t = (row = t >> 2, q = t & 3) keeps Bi[row][4*jj + q], jj = 0..15, in registers
    double breg[REG ? 16 : 1];
    int ncols, nn;  // current width of W and number of non-basic columns
    int wrows, vlen;  // rows of W incl. zero padding; length of the m-vectors incl. zero padding
    double cscale;   // max |cost| of the current phase: reduced costs below 1e-9 * cscale in magnitude are noise
    double anorm_w;  // norm of the basis at its last inversion, scale of the polish residual test
    double cond_inf_last;  // ||B||_inf ||B^-1||_inf of the last successful inversion
    // HBM tier: ring of shared-memory stages fed by TMA bulk copies (nullptr: plain loads)
    double* ring;
    unsigned long long* ring_bar;
    int ring_stage_doubles, ring_ns, ring_uses, stream_min_m;
    int* sel;  // row list of the current stream (aliases inb: the flags are dead inside the main loop)
    bool bi_smem;    // tiers 2, 3: Bi lives in shared memory with a quad-friendly row stride
    bool w_loaded;   // REG tier: W holds [A | art] in ORIGINAL column order for the current LP
    // counters (uniform across the CTA)
    int piv1, piv2, nbland, ninv, used_p1, scan_fb, nrepair;
    int max_pivots, refactor_period;
    // pivot trace of one LP (nullptr: off); cur_phase / cur_bland describe the pivot being made
    int* trace_out;
    int trace_cap, cur_phase, cur_bland;
    // ---- cooperative tier: this CTA is `rank` of `G` CTAs that share one LP (state in HBM, see coop_loop) -------
    int G, rank;
    unsigned long long* gbar;     // the group's barrier counter
    unsigned long long epoch;     // barriers passed so far
    double* mail;                 // the group's mailbox: command, arguments, per-CTA argmin records
    double *Bi1, *Tp, *Rs;        // second buffer of the inverse; inversion panel (m x CNB) and pivot-row snapshot
    double *s_y, *s_prow, *s_ae, *s_xb, *s_al, *s_f, *s_r, *s_part;  // shared-memory scratch of this CTA
    int* s_bit;
    double* s_pan;                // shared-memory inversion panel (aliases the scratch above), nullptr: use Tp
    long long prof_t[16];         // leader: clock cycles in solve, main loop, inversion, polish, leader Bland, refactor;
                                  // [6] main-loop calls, [7] polish calls; [8] input checks, [9] warm start, [10] initial
                                  // basis / Phase-I set-up (outside its main loop), [11] repair loop, [12] results,
                                  // [13] main-loop entry / exit (state load, buffer normalisation)

    GM_DEV void trace_pivot(int enter_var, int leave_var) {  // called by ONE thread, before the counters move
        if constexpr (WARM) {
            if (trace_out) {
                const int k = piv1 + piv2;
                if (k < trace_cap) {
                    int* rr = trace_out + 4 * k;
                    rr[0] = cur_phase; rr[1] = enter_var; rr[2] = leave_var; rr[3] = cur_bland;
                }
            }
        }
    }

    GM_DEV static int pow2ceil(int v) {
        int p = 1;
        while (p < v) p <<= 1;
        return p;
    }

    // ---- problem source: [A0 0; G I] of convertToEqualities, subproblem.go:81-139 ------------------
    GM_DEV double src_a(int i, int j) const {
        if (i < m0) return j < n0 ? gm_ldg(A0 + (size_t)i * lda + j) : 0.0;
        const int k = i - m0;
        if (j == bvar[k]) return bsign[k];
        return j == n0 + k ? 1.0 : 0.0;
    }
    GM_DEV double src_c(int j) const { return j < n0 ? gm_ldg(c0 + j) : 0.0; }
    GM_DEV double src_b(int i) const { return i < m0 ? gm_ldg(b0 + i) : brhs[i - m0]; }

    // ---- block-wide reductions (result identical in every thread) ---------------------------------
    // COOP: the scratch has two halves used alternately, so a reduction needs one barrier instead of two (the next
    // reduction writes the other half; by the barrier after that every thread has finished reading this one).
    int red_flip;
    GM_DEV int red_base() {
        if constexpr (COOP) { red_flip ^= 1; return red_flip ? gm_nthreads() : 0; }
        return 0;
    }
    GM_DEV void red_tail_sync() {
        if constexpr (!COOP) gm_sync();
    }
    // first minimum over f(k), NaN skipped, all-NaN -> index 0: floats.MinIdx, floats.go:458-474
    template <class F>
    GM_DEV MinLoc block_argmin(int len, F f) {
        const int t = gm_tid(), T = gm_nthreads();
        double bvv = INFINITY;
        int bi = INT_MAX;
        for (int k = t; k < len; k += T) {
            const double v = f(k);
            if (v == v && (bi == INT_MAX || v < bvv)) { bvv = v; bi = k; }
        }
        for (int d = 16; d >= 1; d >>= 1) {
            const double ov = gm_shfl_xor(bvv, d);
            const int oi = gm_shfl_xor(bi, d);
            if (oi != INT_MAX && (bi == INT_MAX || ov < bvv || (ov == bvv && oi < bi))) { bvv = ov; bi = oi; }
        }
        const int nw = T >> 5;
        const int rb = red_base();
        if ((t & 31) == 0) { red[rb + (t >> 5)] = bvv; redi[rb + (t >> 5)] = bi; }
        gm_sync();
        bvv = red[rb];
        bi = redi[rb];
        for (int w = 1; w < nw; ++w) {
            const double ov = red[rb + w];
            const int oi = redi[rb + w];
            if (oi != INT_MAX && (bi == INT_MAX || ov < bvv || (ov == bvv && oi < bi))) { bvv = ov; bi = oi; }
        }
        red_tail_sync();
        MinLoc out;
        out.v = bvv;
        out.i = bi == INT_MAX ? 0 : bi;
        if (bi == INT_MAX) out.v = NAN;
        return out;
    }

    template <class F>
    GM_DEV double block_sum(int len, F f) {
        const int t = gm_tid(), T = gm_nthreads();
        double s = 0;
        for (int k = t; k < len; k += T) s += f(k);
        for (int d = 16; d >= 1; d >>= 1) s += gm_shfl_xor(s, d);
        const int nw = T >> 5;
        const int rb = red_base();
        if ((t & 31) == 0) red[rb + (t >> 5)] = s;
        gm_sync();
        s = 0;
        for (int w = 0; w < nw; ++w) s += red[rb + w];
        red_tail_sync();
        return s;
    }

    template <class F>
    GM_DEV double block_max(int len, F f) {  // max over f(k) >= 0; NaN propagates as +Inf
        const int t = gm_tid(), T = gm_nthreads();
        double s = 0;
        for (int k = t; k < len; k += T) {
            const double v = f(k);
            s = (v != v) ? INFINITY : fmax(s, v);
        }
        for (int d = 16; d >= 1; d >>= 1) s = fmax(s, gm_shfl_xor(s, d));
        const int nw = T >> 5;
        const int rb = red_base();
        if ((t & 31) == 0) red[rb + (t >> 5)] = s;
        gm_sync();
        s = 0;
        for (int w = 0; w < nw; ++w) s = fmax(s, red[rb + w]);
        red_tail_sync();
        return s;
    }

    template <class F>
    GM_DEV int block_min_int(int len, F f) {  // min over f(k) (ints), INT_MAX when empty
        const int t = gm_tid(), T = gm_nthreads();
        int s = INT_MAX;
        for (int k = t; k < len; k += T) {
            const int v = f(k);
            s = v < s ? v : s;
        }
        for (int d = 16; d >= 1; d >>= 1) {
            const int o = gm_shfl_xor(s, d);
            s = o < s ? o : s;
        }
        const int nw = T >> 5;
        const int rb = red_base();
        if ((t & 31) == 0) redi[rb + (t >> 5)] = s;
        gm_sync();
        s = INT_MAX;
        for (int w = 0; w < nw; ++w) s = redi[rb + w] < s ? redi[rb + w] : s;
        red_tail_sync();
        return s;
    }

    // j fastest: lanes walk the contiguous dimension
    template <class F>
    GM_DEV void for_each_2d(int nrows, int ncolumns, F f) {
        const int t = gm_tid(), T = gm_nthreads();
        int S = pow2ceil(ncolumns);
        if (S > T) S = T;
        const int G = T / S;
        for (int i = t / S; i < nrows; i += G)
            for (int j = t % S; j < ncolumns; j += S) f(i, j);
    }

    // out[j] = (base ? base[j] : 0) + sgn * sum_i x[i] * M[i*ld + j]   (Dgemv Trans shape, vector.go:515-610)
    // Lanes walk the contiguous dimension (coalesced / conflict free); the reduction dimension is cut in G
    // contiguous row ranges, each walked 8 rows at a time with the 8 loads issued before the FMAs so that
    // an HBM-resident M keeps 8 requests per thread in flight. A block of 8 rows whose x entries are all
    // zero is skipped (Dgemv skips zero x too; duals and FTRAN columns are sparse on slack-heavy bases).
    GM_DEV void matvec_t(double* out, const double* base, double sgn, const double* M, int ld, int nr, int no,
                         const double* x) {
        const int t = gm_tid(), T = gm_nthreads();
        int S = pow2ceil(no);
        if (S > T) S = T;
        const int G = T / S;
        const int lane = t % S, g = t / S;
        int chunk = (nr + G - 1) / G;
        chunk = (chunk + 7) & ~7;
        const int i0 = g * chunk, i1 = (i0 + chunk < nr) ? i0 + chunk : nr;
        for (int j0 = 0; j0 < no; j0 += S) {
            const int j = j0 + lane;
            double a0 = 0, a1 = 0, a2 = 0, a3 = 0;
            if (j < no) {
                const double* col = M + j;
                int i = i0;
                for (; i + 8 <= i1; i += 8) {
                    double xv[8];
                    bool any = false;
#pragma unroll
                    for (int u = 0; u < 8; ++u) { xv[u] = x[i + u]; any |= xv[u] != 0.0; }
                    if (!any) continue;
                    double v[8];
#pragma unroll
                    for (int u = 0; u < 8; ++u) v[u] = col[(size_t)(i + u) * ld];
                    a0 += xv[0] * v[0]; a1 += xv[1] * v[1]; a2 += xv[2] * v[2]; a3 += xv[3] * v[3];
                    a0 += xv[4] * v[4]; a1 += xv[5] * v[5]; a2 += xv[6] * v[6]; a3 += xv[7] * v[7];
                }
                for (; i < i1; ++i) {
                    const double xi = x[i];
                    if (xi != 0.0) a0 += xi * col[(size_t)i * ld];
                }
            }
            const double acc = (a0 + a1) + (a2 + a3);
            if (G == 1) {
                if (j < no) out[j] = (base ? base[j] : 0.0) + sgn * acc;
            } else {  // no <= S here: a single pass over j
                if constexpr (COOP) gm_sync();  // a barrier-less block reduction may still be reading this scratch
                red[t] = acc;
                gm_sync();
                if (t < no) {
                    double sacc = 0;
                    for (int g2 = 0; g2 < G; ++g2) sacc += red[g2 * S + t];
                    out[t] = (base ? base[t] : 0.0) + sgn * sacc;
                }
            }
        }
        gm_sync();
    }

    // out[i] = (base ? base[i] : 0) + sgn * sum_j M[i*ld + j] * x[j]   (one warp per row, 8 loads in flight per lane)
    GM_DEV void matvec_n(double* out, const double* base, double sgn, const double* M, int ld, int no, int nr,
                         const double* x) {
        const int t = gm_tid(), T = gm_nthreads();
        const int warp = t >> 5, lane = t & 31, nw = T >> 5;
        for (int i = warp; i < no; i += nw) {
            double a0 = 0, a1 = 0, a2 = 0, a3 = 0;
            const double* row = M + (size_t)i * ld;
            int j = lane;
            for (; j + 224 < nr; j += 256) {
                double v[8];
#pragma unroll
                for (int u = 0; u < 8; ++u) v[u] = row[j + 32 * u];
                a0 += v[0] * x[j];       a1 += v[1] * x[j + 32];  a2 += v[2] * x[j + 64];  a3 += v[3] * x[j + 96];
                a0 += v[4] * x[j + 128]; a1 += v[5] * x[j + 160]; a2 += v[6] * x[j + 192]; a3 += v[7] * x[j + 224];
            }
            for (; j < nr; j += 32) a0 += row[j] * x[j];
            double acc = (a0 + a1) + (a2 + a3);
            for (int d = 16; d >= 1; d >>= 1) acc += gm_shfl_xor(acc, d);
            if (lane == 0) out[i] = (base ? base[i] : 0.0) + sgn * acc;
        }
        gm_sync();
    }

    // M[i][j] <- (i == l) ? prw[j] : M[i][j] - f[i] * prw[j]   for i, j < mm, and with zero_col >= 0 the old
    // M[i][zero_col] is taken as 0 (the in-place Gauss-Jordan trick). Rows are walked 8 at a time with the
    // 8 loads issued before the stores; a block of 8 rows with all f == 0 (and not holding row l) is skipped.
    GM_DEV void rank1_update(double* M, int ld, int mm, int l, const double* f, const double* prw, int zero_col) {
        const int t = gm_tid(), T = gm_nthreads();
        for (int i0 = 0; i0 < mm; i0 += 8) {
            const int cnt = mm - i0 < 8 ? mm - i0 : 8;
            double fv[8];
            bool any = (l >= i0 && l < i0 + cnt);
#pragma unroll
            for (int u = 0; u < 8; ++u) { fv[u] = u < cnt ? f[i0 + u] : 0.0; any |= fv[u] != 0.0; }
            if (!any) continue;
            for (int j = t; j < mm; j += T) {
                const double pj = prw[j];
                double v[8];
#pragma unroll
                for (int u = 0; u < 8; ++u)
                    if (u < cnt) v[u] = M[(size_t)(i0 + u) * ld + j];
                if (j == zero_col) {
#pragma unroll
                    for (int u = 0; u < 8; ++u) v[u] = 0.0;
                }
#pragma unroll
                for (int u = 0; u < 8; ++u) {
                    if (u < cnt) {
                        if (i0 + u == l) M[(size_t)(i0 + u) * ld + j] = pj;
                        else if (fv[u] != 0.0) M[(size_t)(i0 + u) * ld + j] = v[u] - fv[u] * pj;
                    }
                }
            }
        }
        gm_sync();
    }

    // ---- verifyInputs, simplex.go:385-439 ---------------------------------------------------------
    // The REG tier reads A from HBM once: straight into W (which keeps the original column order there), and the
    // tests below read W. The other tiers read A0 where it lies.
    GM_DEV int verify_inputs() {
        const int t = gm_tid(), T = gm_nthreads();
        const int warp = t >> 5, lane = t & 31, nw = T >> 5;
        if constexpr (REG) load_w_reg();
        auto a0 = [&](int i, int j) -> double {
            if constexpr (REG) return W[i * ldw + j];
            else return gm_ldg(A0 + (size_t)i * lda + j);
        };
        // first all-zero row (only root rows can be: a branch row always holds its slack's 1)
        int zr = INT_MAX;
        for (int i = warp; i < m0; i += nw) {
            int nz = 0;
            for (int j = lane; j < n0; j += 32) nz |= (a0(i, j) != 0.0);
            nz = gm_any(nz);
            if (!nz && i < zr) zr = i;
        }
        zr = block_min_int(T, [&](int k) { return k == t ? zr : INT_MAX; });
        if (zr != INT_MAX) return src_b(zr) != 0.0 ? GM_ERR_INFEASIBLE : GM_ERR_ZERO_ROW;
        // first all-zero column (slack columns n0.. are never zero)
        int zc = INT_MAX;
        for (int j = t; j < n0; j += T) {
            int nz = 0;
            for (int i = 0; i < m0 && !nz; ++i) nz = (a0(i, j) != 0.0);
            for (int k = 0; k < L && !nz; ++k) nz = (bvar[k] == j && bsign[k] != 0.0);
            if (!nz && j < zc) zc = j;
        }
        zc = block_min_int(T, [&](int k) { return k == t ? zc : INT_MAX; });
        if (zc != INT_MAX) return src_c(zc) < 0.0 ? GM_ERR_UNBOUNDED : GM_ERR_ZERO_COLUMN;
        return GM_OK;
    }

    // REG tier: W[i][v] = [A0 0; G I][i][v] for v < n, zero rows from m up to wrows. A thread owns one column and
    // eight rows at a time, with the eight loads issued before the stores. Ends with a barrier.
    GM_DEV void load_w_reg() {
        const int t = gm_tid(), T = gm_nthreads();
        int S = pow2ceil(n);
        if (S > T) S = T;
        const int RGn = T / S, col = t % S, rg = t / S;
        for (int v = col; v < n; v += S) {
            for (int i0 = rg * 8; i0 < wrows; i0 += RGn * 8) {
                double w8[8];
#pragma unroll
                for (int u = 0; u < 8; ++u) w8[u] = i0 + u < m ? src_a(i0 + u, v) : 0.0;
#pragma unroll
                for (int u = 0; u < 8; ++u) W[(i0 + u) * ldw + v] = w8[u];
            }
        }
        w_loaded = true;
        gm_sync();
    }

    // ---- W / cost vectors for the current basis (extractColumns :474-488, nonBasicIdx :174-197) -----
    // phase1: costs are e_n (simplex.go:552-553) and column n is the artificial column `art`.
    GM_DEV void build_w(int ncolumns, bool phase1) {
        const int t = gm_tid(), T = gm_nthreads();
        ncols = ncolumns;
        nn = ncols - m;
        for (int j = t; j < ncols; j += T) inb[j] = 0;
        gm_sync();
        for (int p = t; p < m; p += T) inb[basic[p]] = 1;
        gm_sync();
        {   // ascending list of the columns not in the basis: ballot ranks inside a warp, warp totals in redi
            const int lane = t & 31, warp = t >> 5, nw = T >> 5;
            int base = 0;
            for (int j0 = 0; j0 < ncols; j0 += T) {
                const int j = j0 + t;
                const int flag = (j < ncols) && !inb[j];
                const unsigned bal = gm_ballot(flag);
                if (lane == 0) redi[warp] = gm_popc(bal);
                gm_sync();
                int off = base, tot = 0;
                for (int w = 0; w < nw; ++w) {
                    const int c = redi[w];
                    if (w < warp) off += c;
                    tot += c;
                }
                if (flag) nonbasic[off + gm_popc(bal & ((1u << lane) - 1u))] = j;
                base += tot;
                gm_sync();
            }
        }
        if constexpr (REG) {
            if (!w_loaded) load_w_reg();  // scan_basis used W as scratch
            if (phase1)
                for (int i = t; i < wrows; i += T) W[i * ldw + n] = i < m ? art[i] : 0.0;
        } else {
            // thread = (column p, row group): the column's variable is looked up once, rows go eight at a time with the
            // loads issued together (W and A may live in HBM: one latency per 8 rows instead of one per element)
            int S = pow2ceil(ncols);
            if (S > T) S = T;
            const int RGn = T / S, col = t % S, rg = t / S;
            for (int p = col; p < ncols; p += S) {
                const int v = p < m ? basic[p] : nonbasic[p - m];
                for (int i0 = rg * 8; i0 < wrows; i0 += RGn * 8) {
                    double w8[8];
#pragma unroll
                    for (int u = 0; u < 8; ++u) {
                        const int i = i0 + u;
                        w8[u] = i >= m ? 0.0 : ((v == n) ? art[i] : src_a(i, v));
                    }
#pragma unroll
                    for (int u = 0; u < 8; ++u)
                        if (i0 + u < wrows) W[(size_t)(i0 + u) * ldw + p] = w8[u];
                }
            }
        }
        for (int p = t; p < m; p += T) {
            const int v = basic[p];
            cb[p] = phase1 ? (v == n ? 1.0 : 0.0) : src_c(v);
        }
        for (int k = t; k < nn; k += T) {
            const int v = nonbasic[k];
            cn[k] = phase1 ? (v == n ? 1.0 : 0.0) : src_c(v);
        }
        gm_sync();
        cscale = phase1 ? 1.0 : block_max(m > nn ? m : nn, [&](int i) {
            return fmax(i < m ? fabs(cb[i]) : 0.0, i < nn ? fabs(cn[i]) : 0.0);
        });
    }

    // physical column of W that holds basis position p / non-basic position k
    GM_DEV int wcol_b(int p) const { return REG ? basic[p] : p; }
    GM_DEV int wcol_n(int k) const { return REG ? nonbasic[k] : m + k; }

    // out[i] = base[i] + sgn * sum_p B[i][p] x[p]   (B = basic columns of W)
    GM_DEV void basis_mul(double* out, const double* base, double sgn, const double* x) {
        if constexpr (REG) {
            const int t = gm_tid(), row = t >> 2, q = t & 3;
            double a = 0;
#pragma unroll
            for (int jj = 0; jj < 16; ++jj) {
                const int p = 4 * jj + q;
                if (p < m) a += W[row * ldw + basic[p]] * x[p];
            }
            a += gm_shfl_xor(a, 1);
            a += gm_shfl_xor(a, 2);
            if (q == 0 && row < m) out[row] = base[row] + sgn * a;
            gm_sync();
        } else {
            matvec_n(out, base, sgn, W, ldw, m, m, x);
        }
    }
    // out[p] = base[p] + sgn * sum_i x[i] B[i][p]
    GM_DEV void basis_mul_t(double* out, const double* base, double sgn, const double* x) {
        if constexpr (REG) {
            const int t = gm_tid(), p = t >> 2, q = t & 3;
            const double* wc = W + (p < m ? basic[p] : 0) + q * ldw;
            double a = 0;
#pragma unroll
            for (int ii = 0; ii < 16; ++ii) a += x[4 * ii + q] * wc[(4 * ii) * ldw];
            a += gm_shfl_xor(a, 1);
            a += gm_shfl_xor(a, 2);
            if (q == 0 && p < m) out[p] = base[p] + sgn * a;
            gm_sync();
        } else {
            matvec_t(out, base, sgn, W, ldw, m, m, x);
        }
    }

    // =================================================================================================
    // Basis-inverse storage. Generic tiers: Bi is an m x ldb array (shared memory or HBM). REG tier:
    // registers, with the Bi slot of the workspace used as a 64 x 68 staging tile.
    // =================================================================================================
    GM_DEV void reg_dump() {  // staging tile <- registers (ends with a barrier)
        const int t = gm_tid(), row = t >> 2, q = t & 3;
#pragma unroll
        for (int jj = 0; jj < (REG ? 16 : 1); ++jj) Bi[row * ldb + 4 * jj + q] = breg[jj];
        gm_sync();
    }

    // Bi[i][j] = f(i, j) for i, j < m
    template <class F>
    GM_DEV void bi_fill(F f) {
        if constexpr (REG) {
            const int t = gm_tid(), row = t >> 2, q = t & 3;
#pragma unroll
            for (int jj = 0; jj < 16; ++jj) {
                const int col = 4 * jj + q;
                breg[jj] = (row < m && col < m) ? f(row, col) : (row == col ? 1.0 : 0.0);
            }
        } else {
            for_each_2d(m, m, [&](int i, int j) { Bi[(size_t)i * ldb + j] = f(i, j); });
            gm_sync();
        }
    }

    // out[i] = sum_j Bi[i][j] * a[j]; `a` is a workspace vector (REG: zero beyond m, up to 64 entries)
    GM_DEV void bi_mul(double* out, const double* a) {
        if constexpr (REG) {
            const int t = gm_tid(), row = t >> 2, q = t & 3;
            double a0 = 0, a1 = 0;
#pragma unroll
            for (int jj = 0; jj < 16; jj += 2) {
                a0 += breg[jj] * a[4 * jj + q];
                a1 += breg[jj + 1] * a[4 * jj + 4 + q];
            }
            double acc = a0 + a1;
            acc += gm_shfl_xor(acc, 1);
            acc += gm_shfl_xor(acc, 2);
            if (q == 0 && row < m) out[row] = acc;
            gm_sync();
        } else {
            matvec_n(out, nullptr, 1.0, Bi, ldb, m, m, a);
        }
    }

    // out[j] = sum_i x[i] * Bi[i][j]
    GM_DEV void bi_mul_t(double* out, const double* x) {
        if constexpr (REG) reg_dump();
        matvec_t(out, nullptr, 1.0, Bi, ldb, m, m, x);
    }

    // product-form update: row l := row l / al[l]; row i -= al[i] * (new row l). `al` in the workspace.
    GM_DEV void bi_update(int l, const double* alv) {
        const int t = gm_tid(), T = gm_nthreads();
        if constexpr (REG) {
            const int row = t >> 2, q = t & 3;
            const double f = row < m ? alv[row] : 0.0;
            if (row == l) {
#pragma unroll
                for (int jj = 0; jj < 16; ++jj) prow[4 * jj + q] = breg[jj] / f;
            }
            gm_sync();
            if (row == l) {
#pragma unroll
                for (int jj = 0; jj < 16; ++jj) breg[jj] = prow[4 * jj + q];
            } else if (f != 0.0) {
#pragma unroll
                for (int jj = 0; jj < 16; ++jj) breg[jj] -= f * prow[4 * jj + q];
            }
            gm_sync();
        } else {
            const double ap = alv[l];
            for (int j = t; j < m; j += T) prow[j] = Bi[(size_t)l * ldb + j] / ap;
            gm_sync();
            rank1_update(Bi, ldb, m, l, alv, prow, -1);
        }
    }

    // ---- Bi <- inverse of W[:, 0:m] by in-place Gauss-Jordan with partial (row) pivoting -----------
    // Stands in for the LU behind every VecDense.SolveVec (mat/solve.go:110-140, lu.go:63-84,293-325).
    // Returns 0, or 1 when a pivot is exactly zero / non-finite or cond_inf > 1e16 (the two conditions
    // under which LU.Solve reports mat.Condition, lu.go:301,321). *cond1 = ||B||_1 * ||B^-1||_1.
    GM_DEV int invert_basis(double* cond1) {
        if constexpr (REG) return invert_basis_reg(cond1);
        if constexpr (COOP) return invert_basis_coop(cond1);
        const int t = gm_tid(), T = gm_nthreads();
        ninv++;
        for_each_2d(m, m, [&](int i, int j) { Bi[(size_t)i * ldb + j] = W[(size_t)i * ldw + j]; });
        gm_sync();
        const double anorm_inf = block_max(m, [&](int i) {
            double s = 0;
            for (int j = 0; j < m; ++j) s += fabs(Bi[(size_t)i * ldb + j]);
            return s;
        });
        const double anorm_1 = block_max(m, [&](int j) {
            double s = 0;
            for (int i = 0; i < m; ++i) s += fabs(Bi[(size_t)i * ldb + j]);
            return s;
        });
        int singular = 0;
        for (int k = 0; k < m; ++k) {
            // Idamax: first largest |.| in column k at or below the diagonal (dgetf2.go:43-45)
            MinLoc pl = block_argmin(m - k, [&](int q) { return -fabs(Bi[(size_t)(k + q) * ldb + k]); });
            const int p = k + pl.i;
            const double pabs = -pl.v;
            if (!(pabs > 0.0) || pabs == INFINITY) { singular = 1; break; }
            if (p != k) {
                for (int j = t; j < m; j += T) {
                    const double a = Bi[(size_t)k * ldb + j];
                    Bi[(size_t)k * ldb + j] = Bi[(size_t)p * ldb + j];
                    Bi[(size_t)p * ldb + j] = a;
                }
                gm_sync();
            }
            if (t == 0) ipiv[k] = p;
            const double pv = Bi[(size_t)k * ldb + k];
            for (int i = t; i < m; i += T) t1[i] = Bi[(size_t)i * ldb + k];
            for (int j = t; j < m; j += T) prow[j] = (j == k ? 1.0 : Bi[(size_t)k * ldb + j]) / pv;
            gm_sync();
            rank1_update(Bi, ldb, m, k, t1, prow, k);
        }
        if (singular) {
            *cond1 = INFINITY;
            return 1;
        }
        // (PA)^-1 P : undo the row interchanges as column interchanges, last first
        for (int k = m - 1; k >= 0; --k) {
            const int p = ipiv[k];
            if (p != k) {
                for (int i = t; i < m; i += T) {
                    const double a = Bi[(size_t)i * ldb + k];
                    Bi[(size_t)i * ldb + k] = Bi[(size_t)i * ldb + p];
                    Bi[(size_t)i * ldb + p] = a;
                }
                gm_sync();
            }
        }
        const double inorm_inf = block_max(m, [&](int i) {
            double s = 0;
            for (int j = 0; j < m; ++j) s += fabs(Bi[(size_t)i * ldb + j]);
            return s;
        });
        const double inorm_1 = block_max(m, [&](int j) {
            double s = 0;
            for (int i = 0; i < m; ++i) s += fabs(Bi[(size_t)i * ldb + j]);
            return s;
        });
        *cond1 = anorm_1 * inorm_1;
        anorm_w = fmax(anorm_1, anorm_inf);
        const double cond_inf = anorm_inf * inorm_inf;
        cond_inf_last = cond_inf;
        if (!(cond_inf <= GM_CONDITION_TOL)) return 1;
        return 0;
    }

    // sum_{i < m} |M[i * ld]| in ascending i: eight loads are issued ahead of their (still sequential) adds
    GM_DEV double col_abs_sum(const double* M, int ld) const {
        double s = 0;
        int i = 0;
        for (; i + 8 <= m; i += 8) {
            double v[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) v[u] = M[(i + u) * ld];
#pragma unroll
            for (int u = 0; u < 8; ++u) s += fabs(v[u]);
        }
        for (; i < m; ++i) s += fabs(M[i * ld]);
        return s;
    }

    // The same Gauss-Jordan inversion with the matrix in registers: two barriers per elimination step,
    // pivot row and displaced row exchanged through prow / t1, column interchanges undone in one pass
    // through the staging tile.
    GM_DEV int invert_basis_reg(double* cond1) {
        const int t = gm_tid(), T = gm_nthreads();
        const int row = t >> 2, q = t & 3, lane = t & 31, warp = t >> 5, nw = T >> 5;
        ninv++;
        bi_fill([&](int i, int j) { return W[i * ldw + basic[j]]; });
        double rs = 0;
#pragma unroll
        for (int jj = 0; jj < (REG ? 16 : 1); ++jj) rs += fabs(breg[jj]);
        rs += gm_shfl_xor(rs, 1);
        rs += gm_shfl_xor(rs, 2);
        if (row >= m) rs = 0.0;
        const double anorm_inf = block_max(T, [&](int k) { return k == t ? rs : 0.0; });
        const double anorm_1 = block_max(m, [&](int j) { return col_abs_sum(W + basic[j], ldw); });
        // Steps k = 4 jj + kq, kq = 0..3, work on columns 4 jj + q, which a rotation of the registers after every
        // fourth step keeps in breg[0], so that every register index is a constant. prow / t1 carry their rows in the
        // same rotated order. Sixteen rotations restore the natural order, also after a singular pivot.
        int singular = 0;
#pragma unroll 1
        for (int jj = 0; jj < 16; ++jj) {
#pragma unroll 1
            for (int kq = 0; kq < 4 && 4 * jj + kq < m && !singular; ++kq) singular = eliminate_reg(4 * jj + kq, kq);
            const double b0 = breg[0];
#pragma unroll
            for (int u = 0; u < (REG ? 15 : 0); ++u) breg[u] = breg[u + 1];
            breg[REG ? 15 : 0] = b0;
        }
        gm_sync();
        if (singular) {
            *cond1 = INFINITY;
            return 1;
        }
        // (PA)^-1 P : the column interchanges compose into one permutation, applied through the tile
        reg_dump();
        if (t == 0) {
            for (int j = 0; j < 64; ++j) cperm[j] = j;
            for (int k = m - 1; k >= 0; --k) {
                const int p = ipiv[k];
                const int a = cperm[k];
                cperm[k] = cperm[p];
                cperm[p] = a;
            }
        }
        gm_sync();
#pragma unroll
        for (int jj = 0; jj < (REG ? 16 : 1); ++jj) breg[jj] = Bi[row * ldb + cperm[4 * jj + q]];
        double is = 0;
#pragma unroll
        for (int jj = 0; jj < (REG ? 16 : 1); ++jj) is += fabs(breg[jj]);
        is += gm_shfl_xor(is, 1);
        is += gm_shfl_xor(is, 2);
        if (row >= m) is = 0.0;
        const double inorm_inf = block_max(T, [&](int k) { return k == t ? is : 0.0; });
        // column sums are permutation invariant
        const double inorm_1 = block_max(m, [&](int j) { return col_abs_sum(Bi + j, ldb); });
        *cond1 = anorm_1 * inorm_1;
        anorm_w = fmax(anorm_1, anorm_inf);
        const double cond_inf = anorm_inf * inorm_inf;
        cond_inf_last = cond_inf;
        if (!(cond_inf <= GM_CONDITION_TOL)) return 1;
        return 0;
    }

    // Elimination step k = 4 jj + kq of invert_basis_reg, with columns 4 jj + q in breg[0] (register slot u holds
    // columns 4 ((u + jj) mod 16) + q, and prow / t1 entry 4 u + q belongs to that column). Returns 1, before touching
    // any register, when the pivot is zero or not finite.
    GM_DEV int eliminate_reg(int k, int kq) {
        const int t = gm_tid(), T = gm_nthreads();
        const int row = t >> 2, q = t & 3, lane = t & 31, warp = t >> 5, nw = T >> 5;
        const bool on_k = q == kq;  // breg[0] of this lane is column k
        const double sel = breg[0];
        double key = (on_k && row >= k && row < m) ? fabs(sel) : -1.0;
        if (key != key) key = INFINITY;
        // Idamax: first largest |.| in column k at or below the diagonal (dgetf2.go:43-45). The bit
        // pattern of a non-negative double is monotone, so two unsigned REDUX.MAX give the maximum
        // and a REDUX.MIN over the rows that hold it gives the first one. key = -1 marks "not a candidate".
        unsigned long long kb = key >= 0.0 ? gm_d2bits(key) : 0ull;
        unsigned hi = (unsigned)(kb >> 32), lo = (unsigned)kb;
        unsigned mh = gm_warp_max_u32(hi);
        unsigned ml = gm_warp_max_u32(hi == mh ? lo : 0u);
        int idx = gm_warp_min_int((key >= 0.0 && hi == mh && lo == ml) ? row : INT_MAX);
        if (lane == 0) { redi[warp] = (int)mh; redi[32 + warp] = (int)ml; redi[64 + warp] = idx; }
        gm_sync();
        hi = (unsigned)redi[lane & (nw - 1)];
        lo = (unsigned)redi[32 + (lane & (nw - 1))];
        idx = redi[64 + (lane & (nw - 1))];
        mh = gm_warp_max_u32(hi);
        ml = gm_warp_max_u32(hi == mh ? lo : 0u);
        idx = gm_warp_min_int((hi == mh && lo == ml) ? idx : INT_MAX);
        key = idx == INT_MAX ? -1.0 : gm_bits2d(((unsigned long long)mh << 32) | ml);
        if (!(key > 0.0) || key == INFINITY) return 1;
        const int p = idx;
        double f = gm_shfl_idx(sel, (lane & ~3) | kq);  // my row's entry in column k
        if (row == p) {
            const double inv = 1.0 / f;
#pragma unroll
            for (int u = 0; u < (REG ? 16 : 1); ++u) prow[4 * u + q] = (u == 0 && on_k ? 1.0 : breg[u]) * inv;
        }
        if (row == k && p != k) {
#pragma unroll
            for (int u = 0; u < (REG ? 16 : 1); ++u) t1[4 * u + q] = breg[u];
        }
        if (t == 0) ipiv[k] = p;
        gm_sync();
        if (row == k) {
#pragma unroll
            for (int u = 0; u < (REG ? 16 : 1); ++u) breg[u] = prow[4 * u + q];
        } else {
            if (row == p) {  // adopt the displaced row k
#pragma unroll
                for (int u = 0; u < (REG ? 16 : 1); ++u) breg[u] = t1[4 * u + q];
                f = t1[kq];  // column k
            }
            if (f != 0.0) {
#pragma unroll
                for (int u = 0; u < (REG ? 16 : 1); ++u) {
                    const double base = (u == 0 && on_k) ? 0.0 : breg[u];
                    breg[u] = base - f * prow[4 * u + q];
                }
            }
        }
        return 0;
    }

    // xb = Bi b ; y = Bi^T cb
    GM_DEV void recompute_xb_y() {
        bi_mul(xb, bv);
        bi_mul_t(y, cb);
    }

    GM_DEV bool xb_feasible() {  // initializeFromBasic's positivity test, simplex.go:459-468
        const int bad = block_min_int(m, [&](int i) { return xb[i] < -GM_INIT_POS_TOL ? i : INT_MAX; });
        return bad == INT_MAX;
    }

    // ---- "polish": what a fresh factorisation would give, at O(m^2) ----------------------------------
    // One or two steps of iterative refinement of xb (B xb = b) and y (B^T y = cb) against the basic
    // columns kept in W[:, 0:m], using the product-form inverse as the approximate solver. Falls back
    // to a full re-inversion when the inverse has drifted too far for refinement to contract.
    GM_DEV int polish() {
        const int t = gm_tid(), T = gm_nthreads();
        // The product-form inverse contracts the error by ||I - Bi B|| per step (1e-10 or better unless it
        // has drifted badly), so two steps land on the accuracy of the residual evaluation itself, which
        // is what a fresh LU solve achieves. A residual that does not collapse sends us to a full
        // re-inversion.
        for (int it = 0; it < 3; ++it) {
            // t1 = b - B xb ; t2 = cb - B^T y
            basis_mul(t1, bv, -1.0, xb);
            basis_mul_t(t2, cb, -1.0, y);
            if (it == 2) break;
            bi_mul(al, t1);     // dx
            bi_mul_t(mv, t2);   // dy
            for (int i = t; i < m; i += T) {
                xb[i] += al[i];
                y[i] += mv[i];
            }
            gm_sync();
        }
        const double rb = block_max(m, [&](int i) { return fabs(t1[i]); });
        const double rc = block_max(m, [&](int i) { return fabs(t2[i]); });
        const double sb = block_max(m, [&](int i) { return fabs(bv[i]) + anorm_w * fabs(xb[i]); }) + 1e-300;
        const double sc = block_max(m > nn ? m : nn, [&](int i) {
            return (i < m ? fabs(cb[i]) + anorm_w * fabs(y[i]) : 0.0) + (i < nn ? fabs(cn[i]) : 0.0);
        }) + 1e-300;
        if (rb <= 1e-13 * sb && rc <= 1e-13 * sc) return GM_OK;
#ifdef GM_DEBUG_EMU
        if (t == 0) printf("polish -> reinversion: rb=%g sb=%g rc=%g sc=%g pivots=%d\n", rb, sb, rc, sc, piv1 + piv2);
#endif
        double cond1;
        if (invert_basis(&cond1)) return GM_ERR_CONDITION;
        recompute_xb_y();
        return GM_OK;
    }

    // ---- the last m columns taken as a permutation matrix (pure slack basis): Bi = B^T ---------------
    GM_DEV bool try_permutation_basis() {
        const int t = gm_tid(), T = gm_nthreads();
        // quick reject on the very last column (dense problems leave here after one round trip)
        if (n - 1 < n0) {
            const double cnt0 = block_sum(m, [&](int i) { return src_a(i, n - 1) != 0.0 ? 1.0 : 0.0; });
            if (cnt0 != 1.0) return false;
        }
        // Non-zeros of the last m columns are counted with one coalesced, fully parallel sweep (inb[p] = count,
        // +1000 for an entry that is not 1; basic[p] = a row holding one), not column by column.
        for (int i = t; i < m; i += T) { ipiv[i] = -1; inb[i] = 0; basic[i] = -1; }
        gm_sync();
        const int nstruct = n0 - (n - m) > 0 ? n0 - (n - m) : 0;  // how many of the m columns are root columns (v < n0)
        // slack columns of branch rows: a single 1 at row m0 + (v - n0) (convertToEqualities)
        for (int p = t; p < m; p += T) {
            const int v = n - 1 - p;
            if (v >= n0) { inb[p] = 1; basic[p] = m0 + (v - n0); }
        }
        gm_sync();
        if (nstruct > 0) {
            const int p0 = m - nstruct;  // positions p0..m-1 hold columns v = n-1-p < n0
            for_each_2d(m, nstruct, [&](int i, int pp) {
                const int p = p0 + pp;
                const double a = src_a(i, n - 1 - p);
                if (a != 0.0) {
                    gm_atomic_add(&inb[p], a == 1.0 ? 1 : 1000);
                    basic[p] = i;
                }
            });
            gm_sync();
        }
        int ok = 1;
        for (int p = t; p < m; p += T) {
            if (inb[p] != 1) ok = 0;
            else ipiv[basic[p]] = p;  // two columns on one row are caught below
        }
        gm_sync();
        for (int p = t; p < m; p += T)
            if (ok && (basic[p] < 0 || ipiv[basic[p]] != p)) ok = 0;
        const int bad = block_min_int(T, [&](int k) { return (k == t && !ok) ? 0 : INT_MAX; });
        if (bad != INT_MAX) return false;
        for (int p = t; p < m; p += T) basic[p] = n - 1 - p;
        gm_sync();
        build_w(n, false);
        // B[:,p] = e_row(p)  =>  B^-1 = B^T : Bi[p][row(p)] = 1, i.e. Bi[i][j] = (ipiv[j] == i)
        bi_fill([&](int i, int j) { return (ipiv[j] == i) ? 1.0 : 0.0; });
        anorm_w = 1.0;
        return true;
    }

    // ---- findLinearlyIndependent, simplex.go:611-637, with mat.Cond(.,1) of the QR factor ----------
    // (matrix.go:284-322, qr.go:23-39: cond = ||R||_1 ||R^-1||_1). Q (m x k) lives in the Bi slot of the
    // workspace, R^-1 in W. Orthogonalisation is classical Gram-Schmidt applied twice; R^-1 and both
    // 1-norms are carried incrementally, so a candidate costs O(mk + k^2) instead of a fresh O(mk^2) QR.
    GM_DEV int scan_basis() {
        const int t = gm_tid(), T = gm_nthreads();
        scan_fb = 1;
        w_loaded = false;
        for_each_2d(m, m, [&](int i, int j) { W[(size_t)i * ldw + j] = 0.0; });
        gm_sync();
        int k = 0;
        double normR = 0, normRinv = 0;
        for (int v = n - 1; v >= 0 && k < m; --v) {
            for (int i = t; i < m; i += T) t1[i] = src_a(i, v);
            gm_sync();
            if (k > 0) {
                matvec_t(t2, nullptr, 1.0, Bi, ldb, m, k, t1);   // s  = Q^T v
                matvec_n(t1, t1, -1.0, Bi, ldb, m, k, t2);       // v -= Q s
                matvec_t(prow, nullptr, 1.0, Bi, ldb, m, k, t1); // s2 = Q^T v
                matvec_n(t1, t1, -1.0, Bi, ldb, m, k, prow);     // v -= Q s2
                for (int j = t; j < k; j += T) t2[j] += prow[j];
                gm_sync();
            }
            const double rho = sqrt(block_sum(m, [&](int i) { return t1[i] * t1[i]; }));
            double colR = rho, colRinv = 1.0 / rho;
            if (k > 0) {
                // rho == 0 (or 1/rho overflowing) is an exactly dependent column: cond = +Inf, rejected
                if (!(rho > 0.0) || colRinv == INFINITY) continue;
                colR += block_sum(k, [&](int j) { return fabs(t2[j]); });
                matvec_n(mv, nullptr, -1.0 / rho, W, ldw, k, k, t2);  // u = -R^-1 r / rho
                colRinv += block_sum(k, [&](int j) { return fabs(mv[j]); });
                const double cond = fmax(normR, colR) * fmax(normRinv, colRinv);
                // "not linearly independent" :630-633 (NaN counts as dependent)
                if (colR != colR || colRinv != colRinv || !(cond <= GM_LINDEP_COND_TOL)) continue;
            }
            for (int i = t; i < m; i += T) Bi[(size_t)i * ldb + k] = t1[i] / rho;
            for (int j = t; j < k; j += T) W[(size_t)j * ldw + k] = mv[j];
            if (t == 0) {
                W[(size_t)k * ldw + k] = 1.0 / rho;
                basic[k] = v;
            }
            normR = fmax(normR, colR);
            normRinv = fmax(normRinv, colRinv);
            ++k;
            gm_sync();
        }
        // the scan used the padded vectors as scratch: restore their zero tails (REG tier invariant)
        for (int i = m + t; i < vlen; i += T) { t1[i] = 0.0; t2[i] = 0.0; prow[i] = 0.0; mv[i] = 0.0; }
        gm_sync();
        return k;
    }

    // ---- computeMove, simplex.go:306-342: al = B^-1 a_e, mv = ratios. GM_OK / GM_ERR_UNBOUNDED -------
    GM_DEV int compute_move(int e) {
        const int t = gm_tid(), T = gm_nthreads();
        // a_e is column m+e of W; stage it contiguously (t1) for the row-dot
        {
            const int ce = wcol_n(e);
            for (int i = t; i < m; i += T) t1[i] = W[(size_t)i * ldw + ce];
        }
        gm_sync();
        bi_mul(al, t1);
        // d = -al, |d| < dRoundTol -> 0 ; Min(d) >= 0 -> unbounded ; move_i = xb_i / |d_i| for d_i < 0
        for (int i = t; i < m; i += T) {
            double d = -al[i];
            if (fabs(d) < GM_D_ROUND_TOL) d = 0.0;
            mv[i] = d < 0.0 ? xb[i] / fabs(d) : INFINITY;
            t2[i] = d;
        }
        gm_sync();
        const int anyneg = block_min_int(m, [&](int i) { return t2[i] < 0.0 ? i : INT_MAX; });
        if (anyneg == INT_MAX) return GM_ERR_UNBOUNDED;
        return GM_OK;
    }

    // ---- condition number of the basis with position p replaced by the column staged in t1 -----------------
    // (al = Bi t1 must be current.) The reference factorises the swapped basis from scratch and takes LAPACK's
    // estimate: replaceBland tests mat.Cond(swapped, 1) < 1e16 (simplex.go:369-379), the Phase-I repair loop accepts
    // a column iff LU.Solve does not report mat.Condition, i.e. cond_inf <= 1e16 (simplex.go:589-605, lu.go:301,321).
    // Here both norms are exact: ||B'||.||B'^-1|| with B'^-1 = E Bi read off the product-form update (O(m^2), no
    // factorisation). inf_norm selects the infinity norm, else the 1-norm.
    GM_DEV double swapped_cond(int p, bool inf_norm) {
        if constexpr (REG) reg_dump();
        const double ap = al[p];
        if (!(fabs(ap) > 0.0) || ap != ap) return INFINITY;  // exactly singular: Dgetrf's zero pivot, cond = +Inf
        const double inv = 1.0 / ap;
        double ninv, nb;
        if (!inf_norm) {
            ninv = block_max(m, [&](int j) {
                const double pj = Bi[(size_t)p * ldb + j] * inv;
                double sum = fabs(pj);
                for (int i = 0; i < m; ++i)
                    if (i != p) sum += fabs(Bi[(size_t)i * ldb + j] - al[i] * pj);
                return sum;
            });
            nb = block_max(m, [&](int q) {
                double sum = 0;
                if (q == p) {
                    for (int i = 0; i < m; ++i) sum += fabs(t1[i]);
                } else {
                    const int cq = wcol_b(q);
                    for (int i = 0; i < m; ++i) sum += fabs(W[(size_t)i * ldw + cq]);
                }
                return sum;
            });
        } else {
            ninv = block_max(m, [&](int i) {
                const double f = al[i] * inv;
                double sum = 0;
                for (int j = 0; j < m; ++j) {
                    const double pj = Bi[(size_t)p * ldb + j];
                    sum += fabs(i == p ? pj * inv : Bi[(size_t)i * ldb + j] - f * pj);
                }
                return sum;
            });
            nb = block_max(m, [&](int i) {
                double sum = fabs(t1[i]);
                for (int q = 0; q < m; ++q)
                    if (q != p) sum += fabs(W[(size_t)i * ldw + wcol_b(q)]);
                return sum;
            });
        }
        return ninv * nb;
    }

    // ---- replaceBland, simplex.go:347-383 -----------------------------------------------------------
    // Candidates are the non-basic positions with r <= -blandNegTol in list order; the first whose ratio test gives a
    // non-zero step wins, else the first zero-step leaving position whose swapped basis has cond_1 < 1e16 (exact
    // norms, see swapped_cond). `weak` reports a pivot element at noise level against its column: the caller
    // rebuilds the inverse right after the pivot so that the product form does not carry the division by it.
    GM_DEV int replace_bland(int& l_out, int& e_out, bool& weak) {
        int from = 0;
        weak = false;
        for (;;) {
            const int i = block_min_int(nn - from, [&](int q) { return r[from + q] <= -GM_BLAND_NEG_TOL ? from + q : INT_MAX; });
            if (i == INT_MAX) return GM_ERR_BLAND;
            const int rc = compute_move(i);
            if (rc != GM_OK) return rc;
            MinLoc ml = block_argmin(m, [&](int q) { return mv[q]; });
            if (fabs(ml.v) > GM_BLAND_ZERO_TOL) { l_out = ml.i; e_out = i; return GM_OK; }
            const double dmax = block_max(m, [&](int q) { return fabs(al[q]); });
            int pfrom = 0;
            for (;;) {
                const int p = block_min_int(m - pfrom, [&](int q) { return mv[pfrom + q] <= GM_BLAND_ZERO_TOL ? pfrom + q : INT_MAX; });
                if (p == INT_MAX) break;
                // same shortcut as the cooperative tier: a healthy pivot element cannot push cond_1 of the swapped basis
                // anywhere near 1e16; the exact value is computed only for weak ones
                if (fabs(al[p]) > 1e-6 * dmax || swapped_cond(p, false) < GM_CONDITION_TOL) {
                    l_out = p; e_out = i;
                    weak = !(fabs(al[p]) > 1e-9 * dmax);
                    return GM_OK;
                }
                pfrom = p + 1;
                if (pfrom >= m) break;
            }
            from = i + 1;
            if (from >= nn) return GM_ERR_BLAND;
        }
    }

    // ---- basis change: product-form update of Bi, xb, y; column swap in W (simplex.go:280-292) -------
    GM_DEV void pivot(int l, int e, double re) {
        const int t = gm_tid(), T = gm_nthreads();
        const double theta = xb[l] / al[l];
        gm_sync();
        bi_update(l, al);  // leaves the new row l in prow
        for (int i = t; i < m; i += T) {
            xb[i] = (i == l) ? theta : xb[i] - al[i] * theta;
            y[i] += re * prow[i];
            const double a = W[(size_t)i * ldw + l];
            W[(size_t)i * ldw + l] = W[(size_t)i * ldw + m + e];
            W[(size_t)i * ldw + m + e] = a;
        }
        if (t == 0) {
            const int v = basic[l];
            trace_pivot(nonbasic[e], v);
            basic[l] = nonbasic[e];
            nonbasic[e] = v;
            const double cc = cb[l];
            cb[l] = cn[e];
            cn[e] = cc;
        }
        gm_sync();
    }

    GM_DEV int refactor() {
        double cond1;
        if (invert_basis(&cond1)) return GM_ERR_CONDITION;
        recompute_xb_y();
        return GM_OK;
    }

    // ---- the simplex main loop, simplex.go:233-293. Requires W, Bi, xb, y, cb, cn current. -----------
    // Returns GM_OK (optimal), GM_ERR_UNBOUNDED (caller returns -Inf / nil) or a "break" status
    // (last iterate is still reported, simplex.go:294-301).
    GM_DEV int main_loop(double tol, int phase, bool fresh) {
        if constexpr (REG) return main_loop_reg(tol, phase, fresh);
        if constexpr (COOP) return main_loop_coop(tol, phase, fresh);
        if (bi_smem && gm_nthreads() <= 1024) return main_loop_quad(tol, phase, fresh);
        if (ring != nullptr && m >= stream_min_m && (nn + 2) <= 8 * gm_nthreads() && ((n + 3) & ~1) <= ring_stage_doubles &&
            ((m + 1) & ~1) <= ring_stage_doubles)
            return main_loop_stream(tol, phase, fresh);
        const int t = gm_tid(), T = gm_nthreads();
        int since = 0;
        for (;;) {
            if (piv1 + piv2 >= max_pivots) return GM_ERR_ITERATION_LIMIT;
            // r = cn - an^T y  (:236-243)
            matvec_t(r, cn, -1.0, W + m, ldw, m, nn, y);
            MinLoc rl = block_argmin(nn, [&](int k) { return r[k]; });
            // A reduced cost that is negative only at noise level must be judged with fresh-quality duals, as the
            // reference does every iteration (simplex.go:236): polish first, then decide.
            if (rl.v >= -tol || rl.v != rl.v || (!fresh && rl.v > -1e-9 * cscale)) {  // :247-250
                if (!fresh) {  // confirm optimality with fresh-quality xb and y
                    const int rc = polish();
                    if (rc != GM_OK) return rc;
                    fresh = true;
                    continue;
                }
                return GM_OK;
            }
            int e = rl.i;
            double re = rl.v;
            for (int k = t; k < nn; k += T)
                if (fabs(r[k]) < GM_R_ROUND_TOL) r[k] = 0.0;  // :252-256
            gm_sync();
            int rc = compute_move(e);
            if (rc != GM_OK) return rc;
            MinLoc ml = block_argmin(m, [&](int q) { return mv[q]; });
            int l = ml.i;
            if (ml.v <= 0.0) {  // :268-277
                nbland++;
                bool weak;
                rc = replace_bland(l, e, weak);
                if (rc != GM_OK) return rc;
                re = r[e];
                if (weak) since = refactor_period;
                cur_bland = 1;
            }
            cur_phase = phase;
            pivot(l, e, re);
            cur_bland = 0;
            if (phase == 1) piv1++; else piv2++;
            fresh = false;
            if (++since >= refactor_period) {
                rc = refactor();
                if (rc != GM_OK) return rc;
                fresh = true;
                since = 0;
            }
        }
    }

    // order-preserving map double -> uint64 (-0.0 canonicalised by the caller)
    GM_DEV static unsigned long long ord_key(double v) {
        const unsigned long long u = gm_d2bits(v);
        return (u >> 63) ? ~u : (u | 0x8000000000000000ull);
    }
    GM_DEV static double ord_val(unsigned long long k) {
        return gm_bits2d((k >> 63) ? (k & 0x7fffffffffffffffull) : ~k);
    }
    // Exact first minimum of (value, position) over a warp with three integer REDUX ops: min of the high
    // word of the ordered key, min of the low word among the lanes that match, min position among the
    // lanes that hold the minimum (ties -> lowest position, like floats.MinIdx). Invalid lanes carry
    // (+Inf, INT_MAX); NaN never reaches here.
    GM_DEV static void warp_argmin(double& v, int& i) {
        const unsigned long long kx = ord_key(v + 0.0);
        const unsigned hi = (unsigned)(kx >> 32), lo = (unsigned)kx;
        const unsigned mh = gm_warp_min_u32(hi);
        const unsigned ml = gm_warp_min_u32(hi == mh ? lo : 0xffffffffu);
        i = gm_warp_min_int((hi == mh && lo == ml) ? i : INT_MAX);
        v = ord_val(((unsigned long long)mh << 32) | ml);
    }

    // REG tier main loop: one simplex iteration = three barriers, state in registers, nothing moves in W.
    //   pricing   thread (k = t>>2, q) sums rows i = q (mod 4) of column nonbasic[k] against its register copy
    //             of y, quad-reduces; first-minimum by REDUX inside the warp, through `red` across warps  barrier 1
    //   FTRAN     thread (row, q) dots its 16 registers of Bi with column nonbasic[e] read in place;
    //   ratio     same first-minimum over rows                                                          barrier 2
    //   publish   the quad of row l writes the scaled pivot row (and theta)                              barrier 3
    //   update    16 FMAs on Bi, 16 on y, xb, all in registers; one lane swaps the two list entries
    // xb (per row) and y (per q) are spilled to the workspace only around the rare generic paths.
    GM_DEV int main_loop_reg(double tol, int phase, bool fresh) {
        const int t = gm_tid(), T = gm_nthreads();
        const int row = t >> 2, q = t & 3, lane = t & 31, warp = t >> 5, nw = T >> 5;
        const int s4 = 4 * ldw;
        int since = 0;
        double yreg[REG ? 16 : 1];
        double xbr;
        auto load_state = [&]() {
#pragma unroll
            for (int ii = 0; ii < (REG ? 16 : 1); ++ii) yreg[ii] = y[4 * ii + q];
            xbr = row < m ? xb[row] : 0.0;
        };
        auto store_state = [&]() {
            if (row == 0) {
#pragma unroll
                for (int ii = 0; ii < (REG ? 16 : 1); ++ii) y[4 * ii + q] = yreg[ii];
            }
            if (q == 0 && row < m) xb[row] = xbr;
            gm_sync();
        };
        load_state();
        for (;;) {
            if (piv1 + piv2 >= max_pivots) { store_state(); return GM_ERR_ITERATION_LIMIT; }
            // ---- pricing: r = cn - an^T y, first minimum (:236-250)
            double bestv = INFINITY;
            int besti = INT_MAX;
            for (int k0 = 0; k0 < nn; k0 += 64) {
                if (k0 + 8 * warp >= nn) break;  // warp-uniform: no column of this pass belongs to this warp
                const int k = k0 + row;
                const bool valid = k < nn;
                const double* wc = W + (valid ? nonbasic[k] : 0) + q * ldw;
                double a0 = 0, a1 = 0, a2 = 0, a3 = 0;
#pragma unroll
                for (int ii = 0; ii < (REG ? 16 : 1); ii += 4) {
                    a0 += yreg[ii] * wc[ii * s4];
                    a1 += yreg[ii + 1] * wc[(ii + 1) * s4];
                    a2 += yreg[ii + 2] * wc[(ii + 2) * s4];
                    a3 += yreg[ii + 3] * wc[(ii + 3) * s4];
                }
                double acc = (a0 + a1) + (a2 + a3);
                acc += gm_shfl_xor(acc, 1);
                acc += gm_shfl_xor(acc, 2);
                if (valid) {
                    const double rk = cn[k] - acc;
                    if (q == 0) r[k] = fabs(rk) < GM_R_ROUND_TOL ? 0.0 : rk;  // rounded copy for Bland (:252-256)
                    if (rk == rk && (besti == INT_MAX || rk < bestv)) { bestv = rk; besti = k; }
                }
            }
            if (besti == INT_MAX) bestv = INFINITY;
            warp_argmin(bestv, besti);
            if (lane == 0) { red[warp] = bestv; redi[warp] = besti; }
            gm_sync();  // (1)
            bestv = red[lane & (nw - 1)];
            besti = redi[lane & (nw - 1)];
            warp_argmin(bestv, besti);
            if (besti == INT_MAX || bestv >= -tol || (!fresh && bestv > -1e-9 * cscale)) {
                store_state();
                if (!fresh) {
                    const int rc = polish();
                    if (rc != GM_OK) return rc;
                    fresh = true;
                    load_state();
                    continue;
                }
                return GM_OK;
            }
            int e = besti;
            double re = bestv;
            // ---- FTRAN + ratio test (computeMove :306-342, MinIdx(move) :268)
            double alpha;
            {
                const double* wc = W + nonbasic[e] + q * ldw;
                double a0 = 0, a1 = 0, a2 = 0, a3 = 0;
#pragma unroll
                for (int jj = 0; jj < (REG ? 16 : 1); jj += 4) {
                    a0 += breg[jj] * wc[jj * s4];
                    a1 += breg[jj + 1] * wc[(jj + 1) * s4];
                    a2 += breg[jj + 2] * wc[(jj + 2) * s4];
                    a3 += breg[jj + 3] * wc[(jj + 3) * s4];
                }
                alpha = (a0 + a1) + (a2 + a3);
                alpha += gm_shfl_xor(alpha, 1);
                alpha += gm_shfl_xor(alpha, 2);
            }
            double mvv = INFINITY;
            int mi = INT_MAX;
            if (row < m) {
                double d = -alpha;
                if (fabs(d) < GM_D_ROUND_TOL) d = 0.0;
                mvv = d < 0.0 ? xbr / fabs(d) : INFINITY;
                if (mvv == mvv) mi = row; else mvv = INFINITY;
            }
            warp_argmin(mvv, mi);
            if (lane == 0) { red[32 + warp] = mvv; redi[32 + warp] = mi; }
            gm_sync();  // (2)
            mvv = red[32 + (lane & (nw - 1))];
            mi = redi[32 + (lane & (nw - 1))];
            warp_argmin(mvv, mi);
            if (mi == INT_MAX) mi = 0;
            if (mvv == INFINITY) { store_state(); return GM_ERR_UNBOUNDED; }  // Min(d) >= 0 (:329-331)
            int l = mi;
            if (mvv <= 0.0) {  // :268-277
                nbland++;
                if (q == 0 && row < m) { al[row] = alpha; }
                store_state();
                bool weak;
                const int rc = replace_bland(l, e, weak);
                if (rc != GM_OK) return rc;
                re = r[e];
                alpha = row < m ? al[row] : 0.0;
                if (weak) since = refactor_period;
                if constexpr (WARM) cur_bland = 1;
            }
            // ---- basis change (:280-292)
            if (row == l) {
                const double inv = 1.0 / alpha;
#pragma unroll
                for (int jj = 0; jj < (REG ? 16 : 1); ++jj) prow[4 * jj + q] = breg[jj] * inv;
                if (q == 0) red[64] = xbr * inv;
            }
            gm_sync();  // (3)
            const double theta = red[64];
            {
                // row l itself: breg - (alpha - 1) * (breg / alpha) = breg / alpha, so one FMA form serves every row
                const double f = row == l ? alpha - 1.0 : alpha;
#pragma unroll
                for (int jj = 0; jj < (REG ? 16 : 1); ++jj) {
                    const double pr = prow[4 * jj + q];
                    breg[jj] -= f * pr;
                    yreg[jj] += re * pr;
                }
            }
            xbr = (row == l) ? theta : xbr - alpha * theta;
            // the two list entries and costs swap; the warp that prices position e does it (no barrier needed)
            if (warp == ((e & 63) >> 3)) {
                if (lane == 0) {
                    const int v = basic[l];
                    if constexpr (WARM) { cur_phase = phase; trace_pivot(nonbasic[e], v); }
                    basic[l] = nonbasic[e];
                    nonbasic[e] = v;
                    const double cc = cb[l];
                    cb[l] = cn[e];
                    cn[e] = cc;
                }
                gm_syncwarp();
            }
            if constexpr (WARM) cur_bland = 0;
            if (phase == 1) piv1++; else piv2++;
            fresh = false;
            if (++since >= refactor_period) {
                store_state();
                const int rc = refactor();
                if (rc != GM_OK) return rc;
                fresh = true;
                since = 0;
                load_state();
            }
        }
    }

    // =================================================================================================
    // HBM tier: TMA-staged streaming of W / Bi rows (cp.async.bulk -> mbarrier -> all threads consume)
    // =================================================================================================
    // Streams rows sel[0..nsel) of a row-major HBM matrix, columns [c0, c0 + wcols) (c0 even, wcols even: 16 B
    // alignment), through `ring_ns` stages. One elected thread issues one bulk copy per row; every thread
    // waits on the stage's mbarrier, calls tile(stage, first, count) and releases the stage at a barrier.
    // Returns false if a copy never completes (reported as GM_ERR_CUDA by the caller, never a hang).
    template <class F>
    GM_DEV bool stream_rows(const double* M, int ld, int c0, int wcols, int nsel, F tile) {
        const int t = gm_tid();
        int R = ring_stage_doubles / wcols;
        if (R > 64) R = 64;
        const int ntiles = (nsel + R - 1) / R;
        const unsigned row_bytes = (unsigned)wcols * 8u;
        const int use0 = ring_uses;  // barrier k%ns has completed (use0 + k)/ns phases before this stream... per-stage counters below
        auto issue = [&](int k) {
            if (t == 0) {
                const int first = k * R;
                const int cnt = nsel - first < R ? nsel - first : R;
                const int sidx = (use0 + k) % ring_ns;
                double* st = ring + (size_t)sidx * ring_stage_doubles;
                gm_mbar_expect_tx(ring_bar + sidx, row_bytes * (unsigned)cnt);
                for (int u = 0; u < cnt; ++u)
                    gm_bulk_g2s(st + (size_t)u * wcols, M + (size_t)sel[first + u] * ld + c0, row_bytes, ring_bar + sidx);
            }
        };
        // W / Bi rows were last written with ordinary stores: make them visible to the TMA (async proxy) first
        gm_fence_proxy_async();
        gm_sync();
        const int pre = ntiles < ring_ns ? ntiles : ring_ns;
        for (int k = 0; k < pre; ++k) issue(k);
        bool ok = true;
        for (int k = 0; k < ntiles; ++k) {
            const int g = use0 + k;
            const int sidx = g % ring_ns;
            if (!gm_mbar_wait(ring_bar + sidx, (unsigned)((g / ring_ns) & 1))) ok = false;
            const int first = k * R;
            const int cnt = nsel - first < R ? nsel - first : R;
            tile(ring + (size_t)sidx * ring_stage_doubles, first, cnt);
            gm_sync();  // stage consumed by everybody: it may be refilled
            if (k + ring_ns < ntiles) issue(k + ring_ns);
        }
        ring_uses = use0 + ntiles;
        // a bounded wait that gave up on some threads only must not split the CTA: agree on the verdict
        const int bad = block_min_int(gm_nthreads(), [&](int k) { return (k == t && !ok) ? 0 : INT_MAX; });
        return bad == INT_MAX;
    }

    // Builds sel[] = ascending list of i in [0, count) with pred(i); returns its length (ballot compaction).
    template <class F>
    GM_DEV int select_rows(int count, F pred) {
        const int t = gm_tid(), T = gm_nthreads();
        const int lane = t & 31, warp = t >> 5, nw = T >> 5;
        int base = 0;
        for (int i0 = 0; i0 < count; i0 += T) {
            const int i = i0 + t;
            const int flag = (i < count) && pred(i);
            const unsigned bal = gm_ballot(flag);
            if (lane == 0) redi[warp] = gm_popc(bal);
            gm_sync();
            int off = base, tot = 0;
            for (int w = 0; w < nw; ++w) {
                const int c = redi[w];
                if (w < warp) off += c;
                tot += c;
            }
            if (flag) sel[off + gm_popc(bal & ((1u << lane) - 1u))] = i;
            base += tot;
            gm_sync();
        }
        return base;
    }

    // The simplex main loop of the HBM tier (same decisions as main_loop, simplex.go:233-293). Per pivot:
    //   pricing   rows of W with y_i != 0 stream through the ring; thread j accumulates column j      (m(n-m) words)
    //   FTRAN     a sparse entering column gathers columns of Bi, a dense one streams all of Bi      (m^2 words)
    //   update    only rows with alpha_i != 0 stream in, are updated and stored back coalesced       (2 m^2 words)
    GM_DEV int main_loop_stream(double tol, int phase, bool fresh) {
        const int t = gm_tid(), T = gm_nthreads();
        const int lane = t & 31, warp = t >> 5, nw = T >> 5;
        constexpr int JMAX = 8;
        int since = 0;
        for (;;) {
            if (piv1 + piv2 >= max_pivots) return GM_ERR_ITERATION_LIMIT;
            // ---- pricing: r = cn - an^T y over the non-basic columns [m, m + nn) of W
            {
                const int c0 = m & ~1;              // aligned start: one basic column may ride along
                const int off = m - c0;
                const int wcols = (nn + off + 1) & ~1;
                double acc[JMAX];
#pragma unroll
                for (int jj = 0; jj < JMAX; ++jj) acc[jj] = 0.0;
                const int nsel = select_rows(m, [&](int i) { return y[i] != 0.0; });
                const bool ok = stream_rows(W, ldw, c0, wcols, nsel, [&](const double* st, int first, int cnt) {
                    for (int u = 0; u < cnt; ++u) {
                        const double yi = y[sel[first + u]];
                        const double* rowp = st + (size_t)u * wcols;
#pragma unroll
                        for (int jj = 0; jj < JMAX; ++jj) {
                            const int j = t + jj * T;
                            if (j < wcols) acc[jj] += yi * rowp[j];
                        }
                    }
                });
                if (!ok) return GM_ERR_CUDA;
#pragma unroll
                for (int jj = 0; jj < JMAX; ++jj) {
                    const int k = t + jj * T - off;
                    if (k >= 0 && k < nn) r[k] = cn[k] - acc[jj];
                }
                gm_sync();
            }
            MinLoc rl = block_argmin(nn, [&](int k) { return r[k]; });
            if (rl.v >= -tol || rl.v != rl.v || (!fresh && rl.v > -1e-9 * cscale)) {
                if (!fresh) {
                    const int rc = polish();
                    if (rc != GM_OK) return rc;
                    fresh = true;
                    continue;
                }
                return GM_OK;
            }
            int e = rl.i;
            double re = rl.v;
            for (int k = t; k < nn; k += T)
                if (fabs(r[k]) < GM_R_ROUND_TOL) r[k] = 0.0;  // :252-256
            gm_sync();
            int rc = compute_move_stream(e);
            if (rc != GM_OK) return rc;
            MinLoc ml = block_argmin(m, [&](int q) { return mv[q]; });
            int l = ml.i;
            if (ml.v <= 0.0) {  // :268-277
                nbland++;
                bool weak;
                rc = replace_bland(l, e, weak);
                if (rc != GM_OK) return rc;
                re = r[e];
                if (weak) since = refactor_period;
                cur_bland = 1;
            }
            cur_phase = phase;
            // ---- basis change: only the rows with alpha_i != 0 move
            {
                const double ap = al[l];
                const double theta = xb[l] / ap;
                const double inv = 1.0 / ap;
                for (int j = t; j < m; j += T) prow[j] = Bi[(size_t)l * ldb + j] * inv;
                gm_sync();
                const int mA = (m + 1) & ~1;
                const int nsel = select_rows(m, [&](int i) { return i == l || al[i] != 0.0; });
                const bool ok = stream_rows(Bi, ldb, 0, mA, nsel, [&](const double* st, int first, int cnt) {
                    for (int u = 0; u < cnt; ++u) {
                        const int i = sel[first + u];
                        const double f = al[i];
                        const double* rowp = st + (size_t)u * mA;
                        double* dst = Bi + (size_t)i * ldb;
                        if (i == l) {
                            for (int j = t; j < m; j += T) dst[j] = prow[j];
                        } else {
                            for (int j = t; j < m; j += T) dst[j] = rowp[j] - f * prow[j];
                        }
                    }
                });
                if (!ok) return GM_ERR_CUDA;
                for (int i = t; i < m; i += T) {
                    xb[i] = (i == l) ? theta : xb[i] - al[i] * theta;
                    y[i] += re * prow[i];
                    const double a = W[(size_t)i * ldw + l];
                    W[(size_t)i * ldw + l] = W[(size_t)i * ldw + m + e];
                    W[(size_t)i * ldw + m + e] = a;
                }
                if (t == 0) {
                    const int v = basic[l];
                    trace_pivot(nonbasic[e], v);
                    basic[l] = nonbasic[e];
                    nonbasic[e] = v;
                    const double cc = cb[l];
                    cb[l] = cn[e];
                    cn[e] = cc;
                }
                gm_sync();
            }
            cur_bland = 0;
            if (phase == 1) piv1++; else piv2++;
            fresh = false;
            if (++since >= refactor_period) {
                rc = refactor();
                if (rc != GM_OK) return rc;
                fresh = true;
                since = 0;
            }
            (void)lane; (void)warp; (void)nw;
        }
    }

    // computeMove for the HBM tier: al = Bi a_e with a_e = column m+e of W.
    GM_DEV int compute_move_stream(int e) {
        const int t = gm_tid(), T = gm_nthreads();
        const int lane = t & 31, warp = t >> 5, nw = T >> 5;
        for (int i = t; i < m; i += T) t1[i] = W[(size_t)i * ldw + m + e];
        gm_sync();
        const int nz = select_rows(m, [&](int i) { return t1[i] != 0.0; });
        if (nz * 4 <= m) {
            // sparse column (a slack has one entry): al = sum_j a_j Bi[:, j], one strided gather per non-zero
            for (int i = t; i < m; i += T) {
                double acc = 0;
                const double* rowp = Bi + (size_t)i * ldb;
                for (int u = 0; u < nz; ++u) {
                    const int j = sel[u];
                    acc += rowp[j] * t1[j];
                }
                al[i] = acc;
            }
            gm_sync();
        } else {
            const int mA = (m + 1) & ~1;
            for (int i = t; i < m; i += T) sel[i] = i;
            gm_sync();
            const bool ok = stream_rows(Bi, ldb, 0, mA, m, [&](const double* st, int first, int cnt) {
                for (int u = warp; u < cnt; u += nw) {
                    const double* rowp = st + (size_t)u * mA;
                    double a0 = 0, a1 = 0;
                    int j = lane;
                    for (; j + 32 < m; j += 64) {
                        a0 += rowp[j] * t1[j];
                        a1 += rowp[j + 32] * t1[j + 32];
                    }
                    if (j < m) a0 += rowp[j] * t1[j];
                    double acc = a0 + a1;
                    for (int d = 16; d >= 1; d >>= 1) acc += gm_shfl_xor(acc, d);
                    if (lane == 0) al[first + u] = acc;
                }
            });
            if (!ok) return GM_ERR_CUDA;
        }
        for (int i = t; i < m; i += T) {
            double d = -al[i];
            if (fabs(d) < GM_D_ROUND_TOL) d = 0.0;
            mv[i] = d < 0.0 ? xb[i] / fabs(d) : INFINITY;
            t2[i] = d;
        }
        gm_sync();
        const int anyneg = block_min_int(m, [&](int i) { return t2[i] < 0.0 ? i : INT_MAX; });
        if (anyneg == INT_MAX) return GM_ERR_UNBOUNDED;
        return GM_OK;
    }

    // ---- warm start: parent's optimal basis plus the slack of the new branch row ------------------------
    // B' = [B 0; g 1] with g = the new row restricted to the basic columns (one entry, +-1, at the branched
    // variable if it is basic), so B'^-1 = [B^-1 0; -g B^-1 1] is read off the parent's inverse without any
    // factorisation. The child is primal infeasible in the new row only; Phase I / II then need a few pivots.
    GM_DEV bool warm_start(const BatchParams& P, int lp) {
        const int t = gm_tid(), T = gm_nthreads();
        if (!P.warm_parent || L < 1) return false;
        const int par = P.warm_parent[lp];
        if (par < 0) return false;
        const int mp = m - 1;
        const long long* pb = P.warm_basis + (size_t)par * mp;
        const double* pbi = P.warm_bi + (size_t)par * mp * mp;
        const int bad = block_min_int(mp, [&](int p) { return (pb[p] < 0 || pb[p] >= n - 1) ? p : INT_MAX; });
        if (bad != INT_MAX) return false;
        for (int p = t; p < mp; p += T) basic[p] = (int)pb[p];
        if (t == 0) basic[mp] = n - 1;
        gm_sync();
        const int bv_new = bvar[L - 1];
        const double sg = bsign[L - 1];
        const int pstar = block_min_int(mp, [&](int p) { return basic[p] == bv_new ? p : INT_MAX; });
        build_w(n, false);
        bi_fill([&](int i, int j) {
            if (i < mp) return j < mp ? pbi[(size_t)i * mp + j] : 0.0;
            if (j == mp) return 1.0;
            return pstar == INT_MAX ? 0.0 : -sg * pbi[(size_t)pstar * mp + j];
        });
        anorm_w = 1.0;
        return true;
    }

    // Tiers 2-3 main loop: the register tier's schedule with the basis inverse read from shared memory.
    // Thread (r = t>>2, q = t&3) owns columns j = q (mod 4) of row i0 + r for every block of T/4 rows; quads reduce
    // by shuffles, first-minima by REDUX. Four barriers per pivot plus one to stage the entering column.
    GM_DEV int main_loop_quad(double tol, int phase, bool fresh) {
        const int t = gm_tid(), T = gm_nthreads();
        const int rq = t >> 2, q = t & 3, lane = t & 31, warp = t >> 5, nw = T >> 5, RB = T >> 2;
        int since = 0;
        auto cross = [&](const double* rv, const int* ri, double& v, int& i) {
            v = lane < nw ? rv[lane] : INFINITY;
            i = lane < nw ? ri[lane] : INT_MAX;
            warp_argmin(v, i);
        };
        for (;;) {
            if (piv1 + piv2 >= max_pivots) return GM_ERR_ITERATION_LIMIT;
            // ---- pricing: r = cn - an^T y (:236-250)
            double bestv = INFINITY;
            int besti = INT_MAX;
            for (int k0 = 0; k0 < nn; k0 += RB) {
                if (k0 + 8 * warp >= nn) break;  // warp-uniform
                const int k = k0 + rq;
                const bool valid = k < nn;
                const double* wc = W + m + (valid ? k : 0);
                double a0 = 0, a1 = 0;
                int i = q;
                // tier 3 reads W from HBM / L2: eight independent loads per trip, or the walk is one L2 latency per row
                for (; i + 28 < m; i += 32) {
                    double v[8];
#pragma unroll
                    for (int u = 0; u < 8; ++u) v[u] = wc[(size_t)(i + 4 * u) * ldw];
#pragma unroll
                    for (int u = 0; u < 8; u += 2) {
                        a0 += y[i + 4 * u] * v[u];
                        a1 += y[i + 4 * u + 4] * v[u + 1];
                    }
                }
                for (; i + 4 < m; i += 8) {
                    a0 += y[i] * wc[(size_t)i * ldw];
                    a1 += y[i + 4] * wc[(size_t)(i + 4) * ldw];
                }
                if (i < m) a0 += y[i] * wc[(size_t)i * ldw];
                double acc = a0 + a1;
                acc += gm_shfl_xor(acc, 1);
                acc += gm_shfl_xor(acc, 2);
                if (valid) {
                    const double rk = cn[k] - acc;
                    if (q == 0) r[k] = fabs(rk) < GM_R_ROUND_TOL ? 0.0 : rk;
                    if (rk == rk && (besti == INT_MAX || rk < bestv)) { bestv = rk; besti = k; }
                }
            }
            if (besti == INT_MAX) bestv = INFINITY;
            warp_argmin(bestv, besti);
            if (lane == 0) { red[warp] = bestv; redi[warp] = besti; }
            gm_sync();  // (1)
            cross(red, redi, bestv, besti);
            if (besti == INT_MAX || bestv >= -tol || (!fresh && bestv > -1e-9 * cscale)) {
                gm_sync();
                if (!fresh) {
                    const int rc = polish();
                    if (rc != GM_OK) return rc;
                    fresh = true;
                    continue;
                }
                return GM_OK;
            }
            int e = besti;
            double re = bestv;
            // ---- entering column staged once, then FTRAN + ratio test (:306-342, :268)
            for (int i = t; i < m; i += T) t1[i] = W[(size_t)i * ldw + m + e];
            gm_sync();  // (2)
            double mvv = INFINITY;
            int mi = INT_MAX;
            for (int i0 = 0; i0 < m; i0 += RB) {
                if (i0 + 8 * warp >= m) break;  // warp-uniform
                const int i = i0 + rq;
                const bool valid = i < m;
                const double* brow = Bi + (size_t)(valid ? i : 0) * ldb;
                double a0 = 0, a1 = 0;
                int j = q;
                for (; j + 4 < m; j += 8) {
                    a0 += brow[j] * t1[j];
                    a1 += brow[j + 4] * t1[j + 4];
                }
                if (j < m) a0 += brow[j] * t1[j];
                double alpha = a0 + a1;
                alpha += gm_shfl_xor(alpha, 1);
                alpha += gm_shfl_xor(alpha, 2);
                if (valid) {
                    double d = -alpha;
                    if (fabs(d) < GM_D_ROUND_TOL) d = 0.0;
                    double mvi = d < 0.0 ? xb[i] / fabs(d) : INFINITY;
                    if (q == 0) { al[i] = alpha; mv[i] = mvi; }
                    if (mvi == mvi && (mi == INT_MAX || mvi < mvv)) { mvv = mvi; mi = i; }
                }
            }
            if (mi == INT_MAX) mvv = INFINITY;
            warp_argmin(mvv, mi);
            if (lane == 0) { red[32 + warp] = mvv; redi[32 + warp] = mi; }
            gm_sync();  // (3)
            cross(red + 32, redi + 32, mvv, mi);
            if (mi == INT_MAX) mi = 0;
            if (mvv == INFINITY) { gm_sync(); return GM_ERR_UNBOUNDED; }
            int l = mi;
            if (mvv <= 0.0) {  // :268-277
                nbland++;
                gm_sync();
                bool weak;
                const int rc = replace_bland(l, e, weak);
                if (rc != GM_OK) return rc;
                re = r[e];
                if (weak) since = refactor_period;
                cur_bland = 1;
            }
            cur_phase = phase;
            // ---- basis change (:280-292)
            const double ap = al[l];
            const double inv = 1.0 / ap;
            const double theta = xb[l] * inv;
            for (int j = t; j < m; j += T) prow[j] = Bi[(size_t)l * ldb + j] * inv;
            gm_sync();  // (4)
            for (int i0 = 0; i0 < m; i0 += RB) {
                if (i0 + 8 * warp >= m) break;
                const int i = i0 + rq;
                if (i < m) {
                    double* brow = Bi + (size_t)i * ldb;
                    if (i == l) {
                        for (int j = q; j < m; j += 4) brow[j] = prow[j];
                    } else {
                        const double f = al[i];
                        if (f != 0.0)
                            for (int j = q; j < m; j += 4) brow[j] -= f * prow[j];
                    }
                }
            }
            for (int i = t; i < m; i += T) {
                xb[i] = (i == l) ? theta : xb[i] - al[i] * theta;
                y[i] += re * prow[i];
                const double a = W[(size_t)i * ldw + l];
                W[(size_t)i * ldw + l] = W[(size_t)i * ldw + m + e];
                W[(size_t)i * ldw + m + e] = a;
            }
            if (t == 0) {
                const int v = basic[l];
                trace_pivot(nonbasic[e], v);
                basic[l] = nonbasic[e];
                nonbasic[e] = v;
                const double cc = cb[l];
                cb[l] = cn[e];
                cn[e] = cc;
            }
            cur_bland = 0;
            if (phase == 1) piv1++; else piv2++;
            fresh = false;
            gm_sync();  // (5)
            if (++since >= refactor_period) {
                const int rc = refactor();
                if (rc != GM_OK) return rc;
                fresh = true;
                since = 0;
            }
        }
    }

    // =================================================================================================
    // Cooperative tier (COOP): G CTAs of ONE cooperative launch share one LP.
    //
    // Why: with fewer LPs than SMs (one large LP - BASELINE config 4 -, the narrow first waves of every B&B) one CTA
    // per LP leaves the GPU idle and runs the pivot at one SM's bandwidth. Here rank 0 (the leader) runs the solver's
    // control flow exactly as the other tiers do, on state that lives in HBM / L2, and hands the two O(m^2)-per-step
    // pieces to the whole group:
    //   coop_loop     the simplex main loop (simplex.go:233-293): pricing by column tiles of W, FTRAN / ratio test /
    //                 rank-1 update by row blocks of the inverse; two group barriers per pivot
    //   coop_invert   blocked Gauss-Jordan inversion, trailing updates on the FP64 tensor cores (DMMA)
    // Helpers (rank > 0) sit in coop_helper_loop and execute what the leader posts in the group's mailbox.
    // All decisions are computed redundantly from the same records, so the CTAs never disagree on control flow.
    // =================================================================================================
    static constexpr int CNB = 32;          // inversion panel width (a multiple of the 8-wide DMMA tile)
    enum { CMD_EXIT = 0, CMD_MAIN = 1, CMD_INVERT = 2 };
    enum { CR_OPT = 0, CR_UNBOUNDED = 1, CR_BLAND = 2, CR_REFACTOR = 3, CR_ITER = 4, CR_BLAND_FAIL = 5 };
    // mailbox layout (doubles): [0] command, [1..9] arguments, [10] flag; then per-CTA records
    static constexpr int MAIL_HDR = 16;
    GM_DEV double* rec_a(int g) const { return mail + MAIL_HDR + 2 * g; }           // {value, position}
    GM_DEV double* rec_b(int g) const { return mail + MAIL_HDR + 2 * G + 4 * g; }   // {ratio, row, alpha, buffer bit}
    GM_DEV double* rec_n(int g) const { return mail + MAIL_HDR + 6 * G + 2 * g; }   // {inf-norm part, 1-norm part}
    GM_DEV double* rec_c(int g) const { return mail + MAIL_HDR + 8 * G + 4 * g; }   // Bland: {row, alpha, ratio, bit}
    GM_DEV void prof_add(int k, long long t0) {
        if (gm_tid() == 0) prof_t[k] += gm_clock() - t0;
    }
    // adds the time since t0 to category k and restarts the clock (cooperative kernel only: free elsewhere)
    GM_DEV void pmark(int k, long long& t0) {
        if constexpr (COOP) {
            const long long now = gm_clock();
            if (gm_tid() == 0) prof_t[k] += now - t0;
            t0 = now;
        }
    }

    // Group barrier: every CTA of the group arrives, all earlier global writes of the group are visible afterwards.
    GM_DEV void grp_sync() {
        gm_sync();
        if (G > 1) {
            ++epoch;
            if (gm_tid() == 0) {
                // release: the CTA's writes so far (ordered before this by the block barrier) become visible before the
                // arrival is; acquire: nothing after the spin is satisfied from before the last arrival
                gm_red_release_add_u64(gbar, 1ull);
                const unsigned long long target = epoch * (unsigned long long)G;
                while (gm_ld_acquire_u64(gbar) < target) gm_spin_pause();
            }
            gm_sync();
        }
    }

    GM_DEV double* bi_buf(int bit) const { return bit ? Bi1 : Bi; }

    // out[j] (shared memory, j < tw) = sum over rows i < nrows of f(i, M[i][c0 + j]); the tile is walked with lanes
    // along the contiguous dimension and T / S row groups, partials combined through s_part. Ends with a barrier.
    template <class F>
    GM_DEV void col_tile_reduce(const double* M, int ld, int nrows, int c0, int tw, double* out, F f) {
        const int t = gm_tid(), T = gm_nthreads();
        int S = pow2ceil(tw > 0 ? tw : 1);
        if (S > T) S = T;
        const int RG = T / S, col = t % S, rg = t / S;
        for (int cb0 = 0; cb0 < tw; cb0 += S) {
            const int j = cb0 + col;
            double a0 = 0, a1 = 0, a2 = 0, a3 = 0;
            if (j < tw) {
                const double* cp = M + c0 + j;
                int i = rg;
                // 16 independent loads per trip: an HBM-resident tile needs ~40 KB in flight per SM (B200: 6.5 TB/s x
                // ~1 us / 148 SMs), i.e. more than the 8-byte loads of 512 threads can cover with a shallow unroll
                for (; i + 15 * RG < nrows; i += 16 * RG) {
                    double v[16];
#pragma unroll
                    for (int u = 0; u < 16; ++u) v[u] = cp[(size_t)(i + u * RG) * ld];
#pragma unroll
                    for (int u = 0; u < 16; u += 4) {
                        a0 += f(i + u * RG, v[u]);
                        a1 += f(i + (u + 1) * RG, v[u + 1]);
                        a2 += f(i + (u + 2) * RG, v[u + 2]);
                        a3 += f(i + (u + 3) * RG, v[u + 3]);
                    }
                }
                for (; i + 3 * RG < nrows; i += 4 * RG) {
                    const double v0 = cp[(size_t)i * ld], v1 = cp[(size_t)(i + RG) * ld];
                    const double v2 = cp[(size_t)(i + 2 * RG) * ld], v3 = cp[(size_t)(i + 3 * RG) * ld];
                    a0 += f(i, v0); a1 += f(i + RG, v1); a2 += f(i + 2 * RG, v2); a3 += f(i + 3 * RG, v3);
                }
                for (; i < nrows; i += RG) a0 += f(i, cp[(size_t)i * ld]);
            }
            s_part[t] = (a0 + a1) + (a2 + a3);
            gm_sync();
            if (t < S && cb0 + t < tw) {
                double acc = 0;
                for (int g2 = 0; g2 < RG; ++g2) acc += s_part[g2 * S + t];
                out[cb0 + t] = acc;
            }
            gm_sync();
        }
    }

    // Rows [r0, r1) of the inverse: apply the pending rank-1 update (row := row - f * prow, the previous pivot row
    // := prow) writing the OTHER buffer, and, fused in the same pass, alpha_i = row_i . a_e. One warp per
    // (row, column chunk); a row with f == 0 is only read. with_dot = false: update only.
    GM_DEV void coop_rows_pass(int r0, int nr, bool pending, int lprev, bool with_dot) {
        const int t = gm_tid(), T = gm_nthreads();
        const int lane = t & 31, warp = t >> 5, nw = T >> 5;
        int C = nr > 0 ? nw / nr : 1;
        if (C < 1) C = 1;
        int clen = (m + C - 1) / C;
        clen = (clen + 31) & ~31;
        const int npairs = nr * C;
        if (C == 1 && m <= 256) {
            // Short rows, several rows per warp (a wide wave of mid-size LPs, one CTA each): a row is only 1 - 4 loads
            // per lane, so walking the rows one after the other costs one L2 latency per row. Four rows go together:
            // all their loads are issued before the first update, then the four dot products are reduced.
            for (int base = warp; base < nr; base += 4 * nw) {
                double2 v[4][4];
                double fr[4], acc[4];
                bool isl[4], wrr[4], ok[4];
                double* dstr[4];
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const int ri = base + q * nw;
                    ok[q] = ri < nr;
                    const int rr = ok[q] ? ri : base;
                    const int i = r0 + rr;
                    const int bit = s_bit[rr];
                    fr[q] = s_f[rr];
                    isl[q] = pending && i == lprev;
                    wrr[q] = ok[q] && pending && (isl[q] || fr[q] != 0.0);
                    const double* src = bi_buf(bit) + (size_t)i * ldb;
                    dstr[q] = bi_buf(bit ^ 1) + (size_t)i * ldb;
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        const int j = 2 * lane + 64 * k;
                        v[q][k] = (ok[q] && j < m) ? *reinterpret_cast<const double2*>(src + j) : double2{0.0, 0.0};
                    }
                }
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    double a0 = 0, a1 = 0;
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        const int j = 2 * lane + 64 * k;
                        if (j < m) {
                            const bool two = j + 1 < m;  // the row may end on an odd column
                            if (wrr[q]) {
                                const double p0 = s_prow[j], p1 = two ? s_prow[j + 1] : 0.0;
                                v[q][k].x = isl[q] ? p0 : v[q][k].x - fr[q] * p0;
                                v[q][k].y = isl[q] ? p1 : v[q][k].y - fr[q] * p1;
                                if (two) *reinterpret_cast<double2*>(dstr[q] + j) = v[q][k];
                                else dstr[q][j] = v[q][k].x;
                            }
                            if (with_dot) {
                                a0 += v[q][k].x * s_ae[j];
                                if (two) a1 += v[q][k].y * s_ae[j + 1];
                            }
                        }
                    }
                    acc[q] = a0 + a1;
                }
                if (with_dot) {
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        double a = acc[q];
                        for (int d = 16; d >= 1; d >>= 1) a += gm_shfl_xor(a, d);
                        if (lane == 0 && ok[q]) s_part[base + q * nw] = a;
                    }
                }
            }
        } else
        for (int pr = warp; pr < npairs; pr += nw) {
            const int ri = pr / C, ch = pr % C;
            const int i = r0 + ri;
            const int j0 = ch * clen, j1 = (j0 + clen < m) ? j0 + clen : m;
            const int bit = s_bit[ri];
            const double f = s_f[ri];
            const bool is_l = pending && i == lprev;
            const bool wr = pending && (is_l || f != 0.0);
            const double* src = bi_buf(bit) + (size_t)i * ldb;
            double* dst = bi_buf(bit ^ 1) + (size_t)i * ldb;
            double a0 = 0, a1 = 0, a2 = 0, a3 = 0;
            // 16-byte loads, 8 strips of 64 columns per trip (128 B in flight per lane, 64 KB per CTA), all issued before
            // anything depends on them: the HBM-resident case is bound by bytes in flight, not by arithmetic. Rows
            // start 32-byte aligned (ldb is a multiple of 4) and chunks at multiples of 32 columns.
            int j = j0 + 2 * lane;
            for (; j + 448 + 1 < j1; j += 512) {
                double2 v[8];
#pragma unroll
                for (int u = 0; u < 8; ++u) v[u] = *reinterpret_cast<const double2*>(src + j + 64 * u);
                if (wr) {
#pragma unroll
                    for (int u = 0; u < 8; ++u) {
                        const double2 pq = *reinterpret_cast<const double2*>(s_prow + j + 64 * u);
                        v[u].x = is_l ? pq.x : v[u].x - f * pq.x;
                        v[u].y = is_l ? pq.y : v[u].y - f * pq.y;
                        *reinterpret_cast<double2*>(dst + j + 64 * u) = v[u];
                    }
                }
                if (with_dot) {
#pragma unroll
                    for (int u = 0; u < 8; u += 2) {
                        const double2 e0 = *reinterpret_cast<const double2*>(s_ae + j + 64 * u);
                        const double2 e1 = *reinterpret_cast<const double2*>(s_ae + j + 64 * (u + 1));
                        a0 += v[u].x * e0.x; a1 += v[u].y * e0.y;
                        a2 += v[u + 1].x * e1.x; a3 += v[u + 1].y * e1.y;
                    }
                }
            }
            for (; j + 1 < j1; j += 64) {
                double2 v0 = *reinterpret_cast<const double2*>(src + j);
                if (wr) {
                    const double2 pq = *reinterpret_cast<const double2*>(s_prow + j);
                    v0.x = is_l ? pq.x : v0.x - f * pq.x;
                    v0.y = is_l ? pq.y : v0.y - f * pq.y;
                    *reinterpret_cast<double2*>(dst + j) = v0;
                }
                if (with_dot) { a0 += v0.x * s_ae[j]; a1 += v0.y * s_ae[j + 1]; }
            }
            if (j < j1) {  // odd tail: one last column
                double v0 = src[j];
                if (wr) {
                    v0 = is_l ? s_prow[j] : v0 - f * s_prow[j];
                    dst[j] = v0;
                }
                if (with_dot) a0 += v0 * s_ae[j];
            }
            if (with_dot) {
                double acc = (a0 + a1) + (a2 + a3);
                for (int d = 16; d >= 1; d >>= 1) acc += gm_shfl_xor(acc, d);
                if (lane == 0) s_part[pr] = acc;
            }
        }
        gm_sync();
        for (int ri = t; ri < nr; ri += T) {
            if (with_dot) {
                double acc = 0;
                for (int ch = 0; ch < C; ++ch) acc += s_part[ri * C + ch];
                s_al[ri] = acc;
            }
            if (pending && (r0 + ri == lprev || s_f[ri] != 0.0)) s_bit[ri] ^= 1;
        }
        gm_sync();
    }

    // The simplex main loop of the cooperative tier; every CTA of the group runs it with the same arguments.
    // Returns why it stopped (CR_*). State on entry / exit: W, Bi (buffer 0), xb, y, lists, cb, cn in HBM.
    // Per pivot:
    //   pricing   my tile of the non-basic columns against the CTA-local copy of y      -> record A, group barrier
    //   FTRAN     my rows of the inverse . a_e, FUSED with the previous pivot's rank-1 update of those rows
    //             (each row is read once and written once per pivot: 2 m^2 + m (n - m) words)
    //   ratio     first minimum over my rows                                            -> record B, group barrier
    //   update    y, xb, the lists; the rank-1 update itself is deferred to the next FTRAN pass
    // A row of the inverse lives in one of two buffers (s_bit): an update writes the other one, so the pivot row
    // everybody reads is never overwritten in the same pivot and no third barrier is needed.
    GM_DEV int coop_loop(double tol, int phase, bool& fresh, int& since, int& e_out) {
        const int t = gm_tid(), T = gm_nthreads();
        const int r0 = (int)(((long long)rank * m) / G), r1 = (int)(((long long)(rank + 1) * m) / G), nr = r1 - r0;
        const int k0 = (int)(((long long)rank * nn) / G), k1 = (int)(((long long)(rank + 1) * nn) / G), tw = k1 - k0;
        long long tp = gm_clock();
        for (int i = t; i < m; i += T) s_y[i] = y[i];
        for (int i = t; i < nr; i += T) { s_xb[i] = xb[r0 + i]; s_f[i] = 0.0; s_bit[i] = 0; s_al[i] = 0.0; }
        gm_sync();
        pmark(13, tp);
        bool pending = false;
        int lprev = -1, skip = -1, reason;
        double skip_r = 0.0;
        for (;;) {
            if (piv1 + piv2 >= max_pivots) { reason = CR_ITER; break; }
            // ---- pricing: r = cn - an^T y over my tile (:236-250)
            col_tile_reduce(W, ldw, m, m + k0, tw, s_r, [&](int i, double v) { return s_y[i] * v; });
            for (int k = t; k < tw; k += T) {
                // the variable that just left the basis sits at position `skip`; its reduced cost is -r_e / alpha_l
                // analytically (its column is being swapped into place by the row owners right now)
                const double rk = (k0 + k == skip) ? skip_r : cn[k0 + k] - s_r[k];
                s_r[k] = rk;
                r[k0 + k] = fabs(rk) < GM_R_ROUND_TOL ? 0.0 : rk;  // rounded copy for Bland (:252-256)
            }
            gm_sync();
            MinLoc rl = block_argmin(tw, [&](int k) { return s_r[k]; });
            if (t == 0) {
                double* ra = rec_a(rank);
                const bool valid = tw > 0 && rl.v == rl.v;
                ra[0] = valid ? rl.v : INFINITY;
                ra[1] = valid ? (double)(k0 + rl.i) : -1.0;
            }
            grp_sync();  // (A)
            MinLoc best = block_argmin(G, [&](int g) { return rec_a(g)[1] >= 0.0 ? rec_a(g)[0] : NAN; });
            const double bestv = best.v;
            const int besti = bestv == bestv ? (int)rec_a(best.i)[1] : -1;
            if (besti < 0 || bestv >= -tol || (!fresh && bestv > -1e-9 * cscale)) { reason = CR_OPT; break; }
            const int e_price = besti;
            const double re_price = bestv;
            // ---- entering column, then my rows: pending update + FTRAN + ratio test (:306-342, :268)
            for (int i = t; i < m; i += T) s_ae[i] = W[(size_t)i * ldw + m + e_price];
            gm_sync();
            coop_rows_pass(r0, nr, pending, lprev, true);
            pending = false;
            MinLoc ml = block_argmin(nr, [&](int q) {
                double d = -s_al[q];
                if (fabs(d) < GM_D_ROUND_TOL) d = 0.0;
                return d < 0.0 ? s_xb[q] / fabs(d) : INFINITY;
            });
            if (t == 0) {
                double* rb = rec_b(rank);
                const bool valid = nr > 0 && ml.v == ml.v;
                rb[0] = valid ? ml.v : INFINITY;
                rb[1] = valid ? (double)(r0 + ml.i) : -1.0;
                rb[2] = valid ? s_al[ml.i] : 0.0;
                rb[3] = valid ? (double)s_bit[ml.i] : 0.0;
            }
            grp_sync();  // (B)
            MinLoc bl = block_argmin(G, [&](int g) { return rec_b(g)[1] >= 0.0 ? rec_b(g)[0] : NAN; });
            const double mvv = bl.v == bl.v ? bl.v : INFINITY;
            if (mvv == INFINITY) { reason = CR_UNBOUNDED; break; }  // Min(d) >= 0 (:329-331)
            int l = (int)rec_b(bl.i)[1];
            double alpha_l = rec_b(bl.i)[2], theta = mvv;
            int bit_l = (int)rec_b(bl.i)[3];
            int e = e_price;
            double re = re_price;
            bool bland = false;
            if (mvv <= 0.0) {
                // ---- replaceBland (:347-383) by the whole group: candidates in list order, each with its own FTRAN
                // over the row blocks. The step-size test is exact; a zero-step leaving position is accepted here
                // only when its pivot element is healthy (|alpha_p| > 1e-6 max|alpha|, which puts the swapped
                // basis' condition number far below the reference's 1e16 bound); a weaker pivot element hands the
                // decision to the leader, which evaluates the exact condition number (replace_bland).
                nbland++;
                bland = true;
                int from = 0, verdict = -1;  // -1 searching, 0 accepted, else CR_*
                while (verdict < 0) {
                    const int i = block_min_int(nn - from, [&](int q) { return r[from + q] <= -GM_BLAND_NEG_TOL ? from + q : INT_MAX; });
                    if (i == INT_MAX) { verdict = CR_BLAND_FAIL; break; }
                    for (int q = t; q < m; q += T) s_ae[q] = W[(size_t)q * ldw + m + i];
                    gm_sync();
                    coop_rows_pass(r0, nr, false, -1, true);
                    auto ratio = [&](int q) {
                        double d = -s_al[q];
                        if (fabs(d) < GM_D_ROUND_TOL) d = 0.0;
                        return d < 0.0 ? s_xb[q] / fabs(d) : INFINITY;
                    };
                    MinLoc m2 = block_argmin(nr, ratio);
                    const double dm = block_max(nr, [&](int q) { return fabs(s_al[q]); });
                    const int pany = block_min_int(nr, [&](int q) { return ratio(q) <= GM_BLAND_ZERO_TOL ? q : INT_MAX; });
                    if (t == 0) {
                        double* rb = rec_b(rank);
                        const bool valid = nr > 0 && m2.v == m2.v;
                        rb[0] = valid ? m2.v : INFINITY;
                        rb[1] = valid ? (double)(r0 + m2.i) : -1.0;
                        rb[2] = valid ? s_al[m2.i] : 0.0;
                        rb[3] = valid ? (double)s_bit[m2.i] : 0.0;
                        rec_n(rank)[0] = dm;
                        double* rc = rec_c(rank);
                        rc[0] = pany != INT_MAX ? (double)(r0 + pany) : -1.0;
                        rc[1] = pany != INT_MAX ? s_al[pany] : 0.0;
                        rc[2] = pany != INT_MAX ? ratio(pany) : 0.0;
                        rc[3] = pany != INT_MAX ? (double)s_bit[pany] : 0.0;
                    }
                    grp_sync();
                    MinLoc b2 = block_argmin(G, [&](int g) { return rec_b(g)[1] >= 0.0 ? rec_b(g)[0] : NAN; });
                    const double mv2 = b2.v == b2.v ? b2.v : INFINITY;
                    const double dmax = block_max(G, [&](int g) { return rec_n(g)[0]; });
                    const int gp = block_min_int(G, [&](int g) { return rec_c(g)[0] >= 0.0 ? g : INT_MAX; });
                    if (mv2 == INFINITY) { verdict = CR_UNBOUNDED; }
                    else if (fabs(mv2) > GM_BLAND_ZERO_TOL) {
                        l = (int)rec_b(b2.i)[1]; alpha_l = rec_b(b2.i)[2]; bit_l = (int)rec_b(b2.i)[3]; theta = mv2;
                        e = i; verdict = 0;
                    } else if (gp != INT_MAX && fabs(rec_c(gp)[1]) > 1e-6 * dmax) {
                        l = (int)rec_c(gp)[0]; alpha_l = rec_c(gp)[1]; theta = rec_c(gp)[2]; bit_l = (int)rec_c(gp)[3];
                        e = i; verdict = 0;
                    } else if (gp != INT_MAX) {
                        verdict = CR_BLAND;  // weak pivot element: the exact condition test decides (leader)
                    } else {
                        from = i + 1;
                        if (from >= nn) verdict = CR_BLAND_FAIL;
                    }
                    grp_sync();  // the records are rewritten by the next candidate / the next pivot
                }
                if (verdict != 0) { reason = verdict; e_out = e_price; nbland -= (verdict == CR_BLAND); break; }
                re = r[e];
            }
            // ---- basis change (:280-292)
            const double inv = 1.0 / alpha_l;
            {
                const double* prw = bi_buf(bit_l) + (size_t)l * ldb;
                for (int j = t; j < m; j += T) s_prow[j] = prw[j] * inv;
            }
            gm_sync();
            for (int j = t; j < m; j += T) s_y[j] += re * s_prow[j];
            for (int q = t; q < nr; q += T) {
                const int i = r0 + q;
                const double a = s_al[q];
                s_xb[q] = (i == l) ? theta : s_xb[q] - a * theta;
                s_f[q] = a;
                const double wl = W[(size_t)i * ldw + l];
                W[(size_t)i * ldw + l] = s_ae[i];
                W[(size_t)i * ldw + m + e] = wl;
            }
            if (rank == 0 && t == 0) {
                const int v = basic[l];
                cur_phase = phase; cur_bland = bland ? 1 : 0;
                trace_pivot(nonbasic[e], v);
                basic[l] = nonbasic[e];
                nonbasic[e] = v;
                const double cc = cb[l];
                cb[l] = cn[e];
                cn[e] = cc;
            }
            pending = true;
            lprev = l;
            skip = e;
            skip_r = -re * inv;
            if (phase == 1) piv1++; else piv2++;
            fresh = false;
            gm_sync();
            if (++since >= refactor_period) { reason = CR_REFACTOR; break; }
        }
        // ---- hand the state back: finish a deferred update, gather every row in buffer 0, store xb / y
        tp = gm_clock();
        if (pending) coop_rows_pass(r0, nr, true, lprev, false);
        {
            const int lane = t & 31, warp = t >> 5, nw = T >> 5;
            for (int q = warp; q < nr; q += nw) {
                if (!s_bit[q]) continue;
                const double* src = Bi1 + (size_t)(r0 + q) * ldb;
                double* dst = Bi + (size_t)(r0 + q) * ldb;
                for (int j = lane; j < m; j += 32) dst[j] = src[j];
            }
        }
        for (int q = t; q < nr; q += T) xb[r0 + q] = s_xb[q];
        if (rank == 0)
            for (int j = t; j < m; j += T) y[j] = s_y[j];
        grp_sync();
        pmark(13, tp);
        return reason;
    }

    // Leader side of the main loop: posts the loop to the group, handles the rare events itself.
    GM_DEV int main_loop_coop(double tol, int phase, bool fresh) {
        const int t = gm_tid();
        int since = 0;
        for (;;) {
            if (t == 0) {
                mail[0] = CMD_MAIN; mail[1] = tol; mail[2] = phase; mail[3] = fresh ? 1.0 : 0.0; mail[4] = since;
                mail[5] = piv1; mail[6] = piv2; mail[7] = cscale; mail[8] = nn; mail[9] = ncols;
                mail[11] = max_pivots;  // the leader may have raised it (robust passes)
            }
            long long t0 = gm_clock();
            grp_sync();
            int e = 0;
            const int reason = coop_loop(tol, phase, fresh, since, e);
            prof_add(1, t0);
            if (t == 0) prof_t[6]++;
            if (reason == CR_ITER) return GM_ERR_ITERATION_LIMIT;
            if (reason == CR_UNBOUNDED) return GM_ERR_UNBOUNDED;
            if (reason == CR_BLAND_FAIL) return GM_ERR_BLAND;
            if (reason == CR_OPT) {
                if (!fresh) {  // confirm optimality with fresh-quality xb and y, like the other tiers
                    t0 = gm_clock();
                    const int rc = polish();
                    prof_add(3, t0);
                    if (t == 0) prof_t[7]++;
                    if (rc != GM_OK) return rc;
                    fresh = true;
                    continue;
                }
                return GM_OK;
            }
            if (reason == CR_REFACTOR) {
                t0 = gm_clock();
                const int rc = refactor();
                prof_add(5, t0);
                if (rc != GM_OK) return rc;
                fresh = true;
                since = 0;
                continue;
            }
            // CR_BLAND with a weak pivot element: resolved by the leader alone on the state in HBM, with the exact
            // condition test of replace_bland (:268-277, :369-379)
            t0 = gm_clock();
            nbland++;
            int l = 0;
            bool weak;
            int rc = replace_bland(l, e, weak);
            if (rc != GM_OK) return rc;
            const double re = r[e];
            cur_bland = 1;
            cur_phase = phase;
            pivot(l, e, re);
            cur_bland = 0;
            if (phase == 1) piv1++; else piv2++;
            fresh = false;
            if (weak || ++since >= refactor_period) {
                rc = refactor();
                if (rc != GM_OK) return rc;
                fresh = true;
                since = 0;
            }
            prof_add(4, t0);
        }
    }

    // ---- blocked Gauss-Jordan inversion of W[:, 0:m] into Bi, trailing updates by DMMA ---------------------------
    // Same contract as invert_basis (stands in for LU.Factorize + Dgecon, lu.go:63-84). Per panel of CNB columns:
    //   leader   unblocked Gauss-Jordan with first-max row pivoting (Idamax, dgetf2.go:43-45) on the m x CNB panel
    //   all      row interchanges and pivot-row snapshot on my column strip, then
    //            M[:, J] += (T[:, K] - I_K) R   for every column J outside the panel: an (m x CNB)(CNB x m) product on
    //            the FP64 tensor cores, 8-row blocks dealt round-robin to the CTAs, 8-column tiles to the warps
    // Runs in every CTA of the group; only the leader's return value / cond1 are used.
    GM_DEV int coop_invert_body(double* cond1) {
        const int t = gm_tid(), T = gm_nthreads();
        const int lane = t & 31, warp = t >> 5, nw = T >> 5;
        const int r0 = (int)(((long long)rank * m) / G), r1 = (int)(((long long)(rank + 1) * m) / G), nr = r1 - r0;
        double* M = Bi;
        ninv++;
        // copy my rows, norms of B: row sums of my rows, column sums of my column strip
        for (int q = warp; q < nr; q += nw)
            for (int j = lane; j < m; j += 32) M[(size_t)(r0 + q) * ldb + j] = W[(size_t)(r0 + q) * ldw + j];
        grp_sync();
        double anorm_inf, anorm_1, inorm_inf, inorm_1;
        coop_norms(M, r0, nr, anorm_inf, anorm_1);
        int singular = 0;
        const int NBW = s_pan ? 16 : CNB;          // panel width
        const int pld = s_pan ? 17 : CNB;          // row stride of the working panel (padded in shared memory)
        double* pan = s_pan ? s_pan : Tp;
        double* pcol = s_pan ? s_pan + (size_t)m * 17 : t1;      // the eliminated column
        double* prw = s_pan ? pcol + ((m + 3) & ~3) : prow;     // the scaled pivot row of the panel
        for (int kb = 0; kb < m; kb += NBW) {
            const int nbk = m - kb < NBW ? m - kb : NBW;
            if (rank == 0) {
                for_each_2d(m, nbk, [&](int i, int q) { pan[(size_t)i * pld + q] = M[(size_t)i * ldb + kb + q]; });
                gm_sync();
                for (int q = 0; q < nbk && !singular; ++q) {
                    const int k = kb + q;
                    MinLoc pl = block_argmin(m - k, [&](int s2) { return -fabs(pan[(size_t)(k + s2) * pld + q]); });
                    const int p = k + pl.i;
                    const double pabs = -pl.v;
                    if (!(pabs > 0.0) || pabs == INFINITY) { singular = 1; break; }
                    if (p != k) {
                        for (int qq = t; qq < nbk; qq += T) {
                            const double a = pan[(size_t)k * pld + qq];
                            pan[(size_t)k * pld + qq] = pan[(size_t)p * pld + qq];
                            pan[(size_t)p * pld + qq] = a;
                        }
                    }
                    if (t == 0) ipiv[k] = p;
                    gm_sync();
                    const double pv = pan[(size_t)k * pld + q];
                    for (int i = t; i < m; i += T) pcol[i] = pan[(size_t)i * pld + q];
                    for (int qq = t; qq < nbk; qq += T) prw[qq] = (qq == q ? 1.0 : pan[(size_t)k * pld + qq]) / pv;
                    gm_sync();
                    for_each_2d(m, nbk, [&](int i, int qq) {
                        const double base = qq == q ? 0.0 : pan[(size_t)i * pld + qq];
                        pan[(size_t)i * pld + qq] = i == k ? prw[qq] : base - pcol[i] * prw[qq];
                    });
                    gm_sync();
                }
                if (!singular) {
                    // the panel's columns are final; Tp (HBM, row stride NBW) gets T[:, K] - I for the trailing update
                    for_each_2d(m, nbk, [&](int i, int q) {
                        const double v = pan[(size_t)i * pld + q];
                        M[(size_t)i * ldb + kb + q] = v;
                        Tp[(size_t)i * NBW + q] = i == kb + q ? v - 1.0 : v;
                    });
                }
                if (t == 0) mail[10] = singular;
            }
            grp_sync();  // panel done
            singular = (int)mail[10];
            if (singular) break;
            {   // my column strip: row interchanges, then the pivot-row snapshot (column-wise, no barriers needed)
                const int c0 = (int)(((long long)rank * m) / G), c1 = (int)(((long long)(rank + 1) * m) / G);
                for (int j = c0 + t; j < c1; j += T) {
                    if (j >= kb && j < kb + nbk) continue;
                    for (int q = 0; q < nbk; ++q) {
                        const int p = ipiv[kb + q];
                        if (p != kb + q) {
                            const double a = M[(size_t)(kb + q) * ldb + j];
                            M[(size_t)(kb + q) * ldb + j] = M[(size_t)p * ldb + j];
                            M[(size_t)p * ldb + j] = a;
                        }
                    }
                    for (int q = 0; q < nbk; ++q) Rs[(size_t)q * ldb + j] = M[(size_t)(kb + q) * ldb + j];
                }
            }
            grp_sync();  // snapshot done
            {   // trailing update on the tensor cores
                const int nrb = (m + 7) >> 3, ntile = (m + 7) >> 3;
                const int arow = lane >> 2, acol = lane & 3;
                for (int rb = rank; rb < nrb; rb += G) {
                    const int i = rb * 8 + arow;
                    double afr[CNB / 4];
#pragma unroll
                    for (int kk = 0; kk < CNB / 4; ++kk) {
                        const int q = kk * 4 + acol;
                        afr[kk] = (i < m && q < nbk) ? Tp[(size_t)i * NBW + q] : 0.0;
                    }
                    for (int jt = warp; jt < ntile; jt += nw) {
                        const int j0 = jt * 8;
                        if (j0 >= kb && j0 < kb + nbk) continue;  // the panel's own columns are already final
                        const int jc = j0 + 2 * acol;
                        double c0v = (i < m && jc < m) ? M[(size_t)i * ldb + jc] : 0.0;
                        double c1v = (i < m && jc + 1 < m) ? M[(size_t)i * ldb + jc + 1] : 0.0;
                        const int jb = j0 + arow;
#pragma unroll
                        for (int kk = 0; kk < CNB / 4; ++kk) {
                            if (kk * 4 < nbk) {  // warp-uniform: panels narrower than CNB stop early
                                const int q = kk * 4 + acol;
                                const double bfr = (q < nbk && jb < m) ? Rs[(size_t)q * ldb + jb] : 0.0;
                                gm_dmma_8x8x4(c0v, c1v, afr[kk], bfr);
                            }
                        }
                        if (i < m && jc < m) M[(size_t)i * ldb + jc] = c0v;
                        if (i < m && jc + 1 < m) M[(size_t)i * ldb + jc + 1] = c1v;
                    }
                }
            }
            grp_sync();  // update done
        }
        if (singular) {
            if (cond1) *cond1 = INFINITY;
            return 1;
        }
        // (PA)^-1 P : the column interchanges compose into one permutation (leader), applied row by row (all)
        if (rank == 0) {
            int* cp = inb;  // m ints of scratch (dead here: build_w refills it)
            if (t == 0) {
                for (int j = 0; j < m; ++j) cp[j] = j;
                for (int k = m - 1; k >= 0; --k) {
                    const int p = ipiv[k];
                    const int a = cp[k];
                    cp[k] = cp[p];
                    cp[p] = a;
                }
            }
        }
        grp_sync();
        for (int q = 0; q < nr; ++q) {
            double* rowp = M + (size_t)(r0 + q) * ldb;
            for (int j = t; j < m; j += T) s_prow[j] = rowp[j];
            gm_sync();
            for (int j = t; j < m; j += T) rowp[j] = s_prow[inb[j]];
            gm_sync();
        }
        grp_sync();
        coop_norms(M, r0, nr, inorm_inf, inorm_1);
        if (cond1) *cond1 = anorm_1 * inorm_1;
        anorm_w = fmax(anorm_1, anorm_inf);
        const double cond_inf = anorm_inf * inorm_inf;
        cond_inf_last = cond_inf;
        if (!(cond_inf <= GM_CONDITION_TOL)) return 1;
        return 0;
    }

    // ||M||_inf and ||M||_1 of the m x m matrix M (row stride ldb), computed by the whole group: row sums of my rows,
    // column sums of my column strip, combined through the mailbox. One group barrier.
    GM_DEV void coop_norms(const double* M, int r0, int nr, double& ninf, double& n1) {
        const int t = gm_tid(), T = gm_nthreads();
        const int lane = t & 31, warp = t >> 5, nw = T >> 5;
        double pinf = 0.0;
        for (int q = warp; q < nr; q += nw) {
            double sum = 0;
            for (int j = lane; j < m; j += 32) sum += fabs(M[(size_t)(r0 + q) * ldb + j]);
            for (int d = 16; d >= 1; d >>= 1) sum += gm_shfl_xor(sum, d);
            pinf = (sum != sum) ? INFINITY : fmax(pinf, sum);
        }
        pinf = block_max(T, [&](int k) { return k == t ? pinf : 0.0; });
        const int c0 = (int)(((long long)rank * m) / G), c1 = (int)(((long long)(rank + 1) * m) / G);
        col_tile_reduce(M, ldb, m, c0, c1 - c0, s_r, [&](int, double v) { return fabs(v); });
        const double p1 = block_max(c1 - c0, [&](int j) { return s_r[j]; });
        if (t == 0) { rec_n(rank)[0] = pinf; rec_n(rank)[1] = p1; }
        grp_sync();
        ninf = block_max(G, [&](int g) { return rec_n(g)[0]; });
        n1 = block_max(G, [&](int g) { return rec_n(g)[1]; });
        grp_sync();
    }

    GM_DEV int invert_basis_coop(double* cond1) {
        if (gm_tid() == 0) mail[0] = CMD_INVERT;
        const long long t0 = gm_clock();
        grp_sync();
        const int rc = coop_invert_body(cond1);
        prof_add(2, t0);
        return rc;
    }

    // Helpers: execute what the leader posts until it says CMD_EXIT.
    GM_DEV void coop_helper_loop() {
        for (;;) {
            grp_sync();
            const int cmd = (int)mail[0];
            if (cmd == CMD_EXIT) return;
            if (cmd == CMD_MAIN) {
                const double tol = mail[1];
                const int phase = (int)mail[2];
                bool fresh = mail[3] != 0.0;
                int since = (int)mail[4];
                piv1 = (int)mail[5]; piv2 = (int)mail[6]; cscale = mail[7]; nn = (int)mail[8]; ncols = (int)mail[9];
                max_pivots = (int)mail[11];
                int e = 0;
                coop_loop(tol, phase, fresh, since, e);
            } else if (cmd == CMD_INVERT) {
                coop_invert_body(nullptr);
            }
        }
    }
    GM_DEV void coop_post_exit() {
        if (gm_tid() == 0) mail[0] = CMD_EXIT;
        grp_sync();
    }

    // ---- findInitialBasic, simplex.go:492-607. On GM_OK: basic, W (n columns), Bi, xb, y, cb, cn set ---
    GM_DEV int find_initial_basic(bool& fresh, bool warm) {
        const int t = gm_tid(), T = gm_nthreads();
        double cond1 = 0;
        long long tp = 0;
        if constexpr (COOP) tp = gm_clock();
        fresh = !warm;  // an inherited inverse is polished before it is trusted for an optimality verdict
        bool have = warm || try_permutation_basis();
        if (!have) {
            // optimistic: the reverse scan accepts the last m columns whenever that block is comfortably
            // conditioned (every leading sub-block is then at least as well conditioned in the 2-norm)
            for (int p = t; p < m; p += T) basic[p] = n - 1 - p;
            gm_sync();
            build_w(n, false);
            const int sing = invert_basis(&cond1);
            // Every m x k leading block M_k of these columns has cond_2(M_k) <= cond_2(B) (interlacing), the reference
            // tests cond_1 of its k x k QR factor, cond_1(R_k) <= k cond_2(M_k), and cond_2(B)^2 <= cond_1(B) cond_inf(B):
            // if m sqrt(cond_1 cond_inf) <= 1e12 the reverse scan provably accepts all m columns (:611-637).
            have = !sing && (double)m * sqrt(cond1 * cond_inf_last) <= GM_LINDEP_COND_TOL;
        }
        if (!have) {
            const int k = scan_basis();
            if (k != m) return GM_ERR_SINGULAR;
            build_w(n, false);
            invert_basis(&cond1);  // a singular result falls into Phase I like initializeFromBasic's error does
        }
        // y is needed only when this basis is feasible: Phase I recomputes it for its own basis
        bi_mul(xb, bv);
        if (xb_feasible()) {
            bi_mul_t(y, cb);
            return GM_OK;
        }

        // Phase I (:529-556)
        used_p1 = 1;
        MinLoc jm = block_argmin(m, [&](int i) { return xb[i]; });
        const int j = jm.i;
        // a_{n+1} = b - sum_{i != j} a_basic[i]
        for (int i = t; i < m; i += T) t1[i] = 1.0;
        gm_sync();
        if (t == 0) t1[j] = 0.0;
        gm_sync();
        basis_mul(art, bv, -1.0, t1);
        // B' = B with column j := art ; B^-1 art = xb - (1 - e_j)
        for (int i = t; i < m; i += T) al[i] = xb[i] - (i == j ? 0.0 : 1.0);
        gm_sync();
        bi_update(j, al);  // the artificial enters position j
        if (t == 0) basic[j] = n;
        gm_sync();
        build_w(n + 1, true);
        bi_mul(xb, bv);
        fresh = false;
        if (!xb_feasible()) {
            double c1;
            const int sing = invert_basis(&c1);
            if (sing) return GM_PANIC_INITIAL_BASIC;  // simplex.go:155-158
            bi_mul(xb, bv);
            if (!xb_feasible()) return GM_PANIC_INITIAL_BASIC;
            fresh = true;
        }
        bi_mul_t(y, cb);
        pmark(10, tp);
        int rc = main_loop(GM_PHASE1_TOL, 1, fresh);
        if constexpr (COOP) tp = gm_clock();
        if (rc != GM_OK) {
            if (rc == GM_ERR_ITERATION_LIMIT || rc == GM_PANIC_INITIAL_BASIC) return rc;
            return GM_ERR_PHASE1_WRAPPED + rc;  // :557-559
        }
        fresh = true;  // main_loop returns optimal only right after a polish
        const int added = block_min_int(m, [&](int p) { return basic[p] == n ? p : INT_MAX; });
        const double xart = added == INT_MAX ? 0.0 : xb[added];
        if (fabs(xart) > GM_PHASE1_ZERO_TOL) return GM_ERR_INFEASIBLE;  // :563-565
        if (added != INT_MAX) {
            // artificial still basic at level zero: first non-basic column (ascending) that yields a
            // non-singular, feasible basis in its place (:581-606)
            for (int v = t; v <= n; v += T) inb[v] = 0;
            gm_sync();
            for (int p = t; p < m; p += T) inb[basic[p]] = 1;
            gm_sync();
            // One pass over A first: the pivot element of column v in the artificial's row is rho . a_v with rho = row
            // `added` of the inverse. Columns where it is exactly zero (nearly all of them: they do not reach that row)
            // give an exactly singular swapped basis, which the reference rejects one LU at a time (:589-605); marking
            // them here (inb = 2) turns n trial solves of O(m^2) into one O(mn) sweep plus the few real candidates.
            if constexpr (REG) reg_dump();
            for (int j = t; j < m; j += T) t2[j] = Bi[(size_t)added * ldb + j];
            gm_sync();
            for (int v = t; v < n; v += T) {
                if (inb[v]) continue;
                double a0 = 0, a1 = 0, s0 = 0, s1 = 0;  // the dot product and the sum of |products| (its rounding scale)
                int i = 0;
                for (; i + 8 <= m; i += 8) {
                    double w[8];
#pragma unroll
                    for (int u = 0; u < 8; ++u) w[u] = src_a(i + u, v);
#pragma unroll
                    for (int u = 0; u < 8; u += 2) {
                        const double p0 = t2[i + u] * w[u], p1 = t2[i + u + 1] * w[u + 1];
                        a0 += p0; a1 += p1; s0 += fabs(p0); s1 += fabs(p1);
                    }
                }
                for (; i < m; ++i) {
                    const double p0 = t2[i] * src_a(i, v);
                    a0 += p0; s0 += fabs(p0);
                }
                // zero, or pure cancellation noise (an inherited product-form inverse has 1e-17s where a fresh LU has
                // exact zeros): the swapped basis is singular to working precision, cond >= 1e16, rejected either way
                if (fabs(a0 + a1) <= 1e-12 * (s0 + s1)) inb[v] = 2;
            }
            gm_sync();
            bool done = false, weak = false;
            for (int v = 0; v < n && !done; ++v) {
                if (inb[v]) {
                    nrepair += inb[v] == 2;  // counted like the reference's trials
                    continue;
                }
                nrepair++;
                for (int i = t; i < m; i += T) t1[i] = src_a(i, v);
                gm_sync();
                bi_mul(al, t1);
                const double amax = block_max(m, [&](int q) { return fabs(al[q]); });
                const double ap = al[added];
                // initializeFromBasic on the swapped basis (:594-600): LU.Solve fails iff the factor is exactly
                // singular or cond_inf > 1e16 (lu.go:301,321); then the positivity test :459-468. A column that does not
                // reach the artificial's row at all (ap == 0: most of them) makes the swapped basis exactly singular; a
                // healthy pivot element (> 1e-6 of the column) puts its condition number within ~1e12 of the current
                // basis', far from 1e16; only in between is the exact condition number (O(m^2)) worth computing.
                // ... and below 1e-14 of the column it is rounding noise of an exact zero (cond >= 1e14 cond(B)).
                if (!(fabs(ap) > 1e-14 * fmax(1.0, amax))) continue;
                if (!(fabs(ap) > 1e-6 * fmax(1.0, amax)) && !(swapped_cond(added, true) <= GM_CONDITION_TOL)) continue;
                weak = !(fabs(ap) > 1e-9 * fmax(1.0, amax));
                // The artificial sits at level |x| <= 1e-12 = zero by the reference's own test (:563), so the swap does
                // not move the vertex: the reference's fresh solve of the swapped basis returns the same xb (its zeros
                // stay within 1e-16 of zero). Dividing the artificial's rounding noise by the pivot element instead
                // would smear it over the degenerate basics and reject candidate after candidate.
                const double theta = 0.0;
                const int bad = block_min_int(m, [&](int i) {
                    const double nx = (i == added) ? theta : xb[i] - al[i] * theta;
                    return nx < -GM_INIT_POS_TOL ? i : INT_MAX;
                });
                if (bad != INT_MAX) continue;
                bi_update(added, al);
                for (int i = t; i < m; i += T) xb[i] = (i == added) ? theta : xb[i] - al[i] * theta;
                if (t == 0) basic[added] = v;
                gm_sync();
                done = true;
                fresh = false;
            }
            if (!done) return GM_ERR_INFEASIBLE;
            if (weak) {  // the accepted pivot element is noise against its column: do not keep the product form
                build_w(n, false);
                double c1;
                if (invert_basis(&c1)) return GM_ERR_PHASE1_WRAPPED + GM_ERR_CONDITION;
                recompute_xb_y();
                fresh = true;
                return GM_OK;
            }
        }
        pmark(11, tp);
        build_w(n, false);  // Phase II lists: basis positions kept, non-basic ascending again (:174-197)
        bi_mul_t(y, cb);
        pmark(10, tp);
        return GM_OK;
    }

    // ---- robust mode (NOT the reference's behaviour; opt-in, gm_options.robust / GM_BNB_ROBUST) -----------------------
    // On highly degenerate LPs (knapsack children: integer data, many active bound rows) the reference's rule set
    // accepts zero-step Bland pivots on noise-level elements, reaches numerically singular bases (mat.Condition), dead
    // ends (ErrBland) or cycles; GoMILP then panics (tree.go:272). With `robust` such an LP is solved once more with its
    // Phase II on a right-hand side perturbed by ~1e-7 relative (B eps, i.e. every basic variable of the Phase-I vertex
    // moved up), which makes the vertices non-degenerate (every step is strictly positive, so the simplex method
    // cannot cycle and never enters replaceBland); the optimal basis found is then
    // re-evaluated on the TRUE right-hand side and, if that leaves it primal infeasible by a hair, repaired by
    // Phase I / II from that basis. The answer is an optimal vertex of the original LP, confirmed by the usual polish.
    // (Implemented as extra passes of the loop in solve(), so that the phases are not inlined a second time.)
    GM_DEV static bool robust_retryable(int st) {
        return st == GM_ERR_BLAND || st == GM_ERR_CONDITION || st == GM_ERR_ITERATION_LIMIT || st == GM_ERR_LINSOLVE ||
               st == GM_PANIC_INITIAL_BASIC || (st > GM_ERR_PHASE1_WRAPPED && st < GM_ERR_BAD_SHAPE);
    }
    // ---- one LP: simplex(), simplex.go:93-302 -------------------------------------------------------
    GM_DEV void solve(const BatchParams& P, int lp) {
        const int t = gm_tid(), T = gm_nthreads();
        piv1 = piv2 = nbland = ninv = used_p1 = scan_fb = nrepair = 0;
        anorm_w = 0.0;
        w_loaded = false;
        int status = GM_OK;
        double optF = NAN;
        bool have_x = false, have_basis = false, ran_main = false;

        // every padded vector starts as zeros (REG tier reads up to 64 entries)
        for (int i = t; i < vlen; i += T) {
            xb[i] = 0.0; cb[i] = 0.0; y[i] = 0.0; al[i] = 0.0; mv[i] = 0.0; prow[i] = 0.0; art[i] = 0.0;
            t1[i] = 0.0; t2[i] = 0.0;
            bv[i] = i < m ? src_b(i) : 0.0;
        }
        gm_sync();
        long long tp = 0;
        if constexpr (COOP) tp = gm_clock();
        status = verify_inputs();
        pmark(8, tp);
        if (status != GM_OK) {
            optF = status == GM_ERR_UNBOUNDED ? -INFINITY : NAN;
        } else if (m > n) {
            status = GM_ERR_SINGULAR;  // findLinearlyIndependent cannot find m columns (:495-498)
        } else if (m == n) {  // :103-119
            for (int p = t; p < m; p += T) basic[p] = p;
            gm_sync();
            build_w(n, false);
            double c1;
            if (invert_basis(&c1)) {
                status = GM_ERR_SINGULAR;
            } else {
                bi_mul(xb, bv);
                const int neg = block_min_int(m, [&](int i) { return xb[i] < 0.0 ? i : INT_MAX; });
                if (neg != INT_MAX) status = GM_ERR_INFEASIBLE;
                else {
                    optF = block_sum(m, [&](int i) { return xb[i] * cb[i]; });
                    have_x = true;
                }
            }
        } else {
            bool fresh = true;
            bool have_start = false;  // basis, W, Bi, xb, y already in place (caller-supplied initialBasic)
            bool warm = false;
            if (P.initial_basic) {  // :147-160
                const long long* ib = P.initial_basic + (size_t)lp * m;
                const int bad = block_min_int(m, [&](int p) { return (ib[p] < 0 || ib[p] >= n) ? p : INT_MAX; });
                if (bad != INT_MAX) status = GM_ERR_BAD_ARGUMENT;
                else {
                    for (int p = t; p < m; p += T) basic[p] = (int)ib[p];
                    gm_sync();
                    // a repeated index would corrupt the non-basic list: it is a singular basis
                    for (int j = t; j < n; j += T) inb[j] = 0;
                    gm_sync();
                    for (int p = t; p < m; p += T) gm_atomic_add(&inb[basic[p]], 1);
                    gm_sync();
                    const int dup = block_min_int(n, [&](int j2) { return inb[j2] > 1 ? j2 : INT_MAX; });
                    if (dup != INT_MAX) status = GM_PANIC_INITIAL_BASIC;
                    else {
                        build_w(n, false);
                        double c1;
                        if (invert_basis(&c1)) status = GM_PANIC_INITIAL_BASIC;
                        else {
                            recompute_xb_y();
                            if (!xb_feasible()) status = GM_PANIC_INITIAL_BASIC;
                        }
                    }
                }
                have_start = true;
            } else {
                if constexpr (WARM) warm = warm_start(P, lp);
                pmark(9, tp);
            }
            // One pass normally. Robust mode (see above) may add two: (1) the same LP on a perturbed right-hand side,
            // cold; (2) the true right-hand side again, started from the basis (1) ended on. The solver's phases appear
            // once in the code, inside this loop.
            int attempt = 0, cap0 = max_pivots;
            double eps_rel = 1e-7;
            if constexpr (WARM) {
                // robust mode gives the reference's rule set a bounded try: a degenerate LP that has not finished after
                // ~6 (m + n) pivots is stalling (healthy ones need 1 - 3 m), and the perturbed passes are cheaper
                if (P.robust && !P.initial_basic && max_pivots > 6 * (m + n) + 1000) max_pivots = 6 * (m + n) + 1000;
            }
            for (;;) {
                if (!have_start) status = find_initial_basic(fresh, warm);
                if (status == GM_OK) {
                    if constexpr (WARM) {
                        if (attempt == 1) {
                            // Perturb the VERTEX, not b: every basic variable moves up by ~1e-7 relative (b moves by
                            // B eps with it, so that refactorisations and the polish stay consistent). Phase I ran on
                            // the true right-hand side: Gonum's construction pins the basics at 1, and a perturbed b
                            // would put 1e-7-sized entries into the artificial column for the ratio test to pivot on.
                            for (int i = t; i < m; i += T) {
                                const double fr = (double)i * 0.6180339887498949;
                                t1[i] = eps_rel * (1.0 + (fr - floor(fr))) * fmax(1.0, fabs(xb[i]));
                            }
                            gm_sync();
                            basis_mul(bv, bv, 1.0, t1);
                            for (int i = t; i < m; i += T) xb[i] += t1[i];
                            gm_sync();
                            fresh = false;
                        }
                    }
                    // the robust passes stop at reduced costs that are noise against the costs (with the reference's
                    // tol = 0 a value of -1e-17 is a pivot, and near-optimal bases can trade places for ever)
                    status = main_loop(attempt > 0 ? fmax(P.tol, 1e-9 * fmax(1.0, cscale)) : P.tol, 2, fresh);
                    ran_main = true;
                }
                bool again = false;
                if constexpr (WARM) {
                    // a cap the caller set (gm_options.max_pivots > 0) bounds the pivots of all passes together
                    const int user_cap = P.max_pivots > 0 ? P.max_pivots : INT_MAX;
                    const long long fresh_cap = (long long)piv1 + piv2 + 50 * (m + n) + 1000;
                    const int retry_cap = fresh_cap < user_cap ? (int)fresh_cap : user_cap;
                    const bool cap_left = piv1 + piv2 < user_cap;
                    if (P.robust && !P.initial_basic && !(attempt == 0 && warm)) {
                        if (attempt == 0 && robust_retryable(status) && cap_left) {
                            scan_fb |= 2;  // reported in stats[5], bit 1
                            max_pivots = retry_cap;
                            fresh = true; warm = false; ran_main = false;
                            attempt = 1;
                            again = true;
                        } else if (attempt == 1) {
                            for (int i = t; i < m; i += T) bv[i] = src_b(i);
                            gm_sync();
                            if (status == GM_OK) {  // re-evaluate the basis on the true right-hand side
                                fresh = false; warm = true; ran_main = false;   // find_initial_basic(warm): from THIS basis
                                attempt = 2;
                                again = true;
                            }
                        }
                        if (!again && attempt >= 1 && robust_retryable(status) && eps_rel < 1e-4 && cap_left) {
                            eps_rel *= 100.0;  // still stuck: once more from scratch with a coarser perturbation
                            max_pivots = retry_cap;
                            fresh = true; warm = false; ran_main = false;
                            attempt = 1;
                            again = true;
                        }
                    }
                }
                if (!again) break;
            }
            max_pivots = cap0;
            if (attempt > 0) warm = false;
            // A warm start follows a different pivot path than the cold solve; if that path dies (ill-conditioned
            // basis, Bland dead end, iteration cap, unbounded ray at noise level) the engine re-solves the node from
            // scratch in a follow-up launch (engine.cu: gm_solve_wave_warm, bnb_device.cu).
            if (warm && status != GM_OK && status != GM_ERR_INFEASIBLE) {
                status = GM_ERR_WARM_RETRY;
                ran_main = false;
            }
            if (ran_main) {
                if (status == GM_ERR_UNBOUNDED) {
                    optF = -INFINITY;  // :260-263
                } else {
                    optF = block_sum(m, [&](int i) { return cb[i] * xb[i]; });  // :296
                    have_x = true;
                    have_basis = true;
                }
            } else if (status == GM_ERR_UNBOUNDED) {
                optF = -INFINITY;
            }
        }

        // ---- results ----
        if constexpr (COOP) tp = gm_clock();
        double* xo = P.x + (size_t)lp * P.x_stride;
        for (int j = t; j < P.x_len; j += T) xo[j] = 0.0;
        gm_sync();
        if (have_x) {
            for (int p = t; p < m; p += T) {
                const int v = basic[p];
                if (v < P.x_len) xo[v] = xb[p];
            }
        }
        if (P.basis) {
            long long* bo = P.basis + (size_t)lp * m;
            const bool keep = have_basis && !(WARM && P.bi_out && status != GM_OK);
            for (int p = t; p < m; p += T) bo[p] = keep ? (long long)basic[p] : -1;
        }
        if (WARM && P.bi_out && have_basis && status == GM_OK) {
            double* out = P.bi_out + (size_t)lp * m * m;
            if constexpr (REG) {
                const int row = t >> 2, q = t & 3;
#pragma unroll
                for (int jj = 0; jj < 16; ++jj) {
                    const int col = 4 * jj + q;
                    if (row < m && col < m) out[(size_t)row * m + col] = breg[jj];
                }
            } else {
                for_each_2d(m, m, [&](int i, int j) { out[(size_t)i * m + j] = Bi[(size_t)i * ldb + j]; });
            }
        }
        if (t == 0) {
            P.status[lp] = status;
            P.optF[lp] = optF;
            if (P.stats) {
                int* s = P.stats + (size_t)lp * 8;
                s[0] = piv1; s[1] = piv2; s[2] = nbland; s[3] = ninv;
                s[4] = used_p1; s[5] = scan_fb; s[6] = nrepair; s[7] = have_x ? 1 : 0;
            }
        }
        gm_sync();
        pmark(12, tp);
    }

    // ---- binding to the workspace (once per CTA: the shape is a launch constant) and to one LP ---------
    GM_DEV void bind_workspace(const BatchParams& P, double* wbase, double* bibase, double* small,
                               double* ring_base = nullptr, unsigned long long* bars = nullptr) {
        G = 1; rank = 0; gbar = nullptr; epoch = 0; mail = nullptr; red_flip = 0;
        ring = ring_base; ring_bar = bars; ring_ns = P.ring_stages; ring_stage_doubles = P.ring_stage_bytes / 8;
        ring_uses = 0;
        stream_min_m = P.stream_min_m;
        m0 = P.m0; n0 = P.n0; L = P.L; lda = P.lda;
        m = m0 + L; n = n0 + L;
        const WsLayout w = ws_layout(m, n, gm_nthreads(), REG, P.hbm_layout != 0, P.tier == 2 || P.tier == 3);
        bi_smem = !REG && (P.tier == 2 || P.tier == 3);
        ldw = w.ldw; ldb = w.ldb; wrows = w.wrows; vlen = w.vlen;
        W = wbase; Bi = bibase;
        xb = small + w.xb; cb = small + w.cb; y = small + w.y; al = small + w.al;
        mv = small + w.mv; bv = small + w.bv; prow = small + w.prow; art = small + w.art; t1 = small + w.t1;
        t2 = small + w.t2; cn = small + w.cn; r = small + w.r; red = small + w.red;
        int* iw = reinterpret_cast<int*>(small + w.small_doubles);
        basic = iw + w.basic; nonbasic = iw + w.nonbasic; inb = iw + w.inb; redi = iw + w.redi; ipiv = iw + w.ipiv;
        cperm = iw + w.cperm;
        sel = inb;
        max_pivots = P.max_pivots > 0 ? P.max_pivots : 50 * (m + n) + 1000;
        refactor_period = P.refactor_period > 0 ? P.refactor_period : (P.hbm_layout && 2 * m > 100 ? 2 * m : 100);
    }
    GM_DEV void bind_lp(const BatchParams& P, int lp) {
        c0 = P.c + (size_t)lp * P.c_stride;
        A0 = P.A + (size_t)lp * P.A_stride;
        b0 = P.b + (size_t)lp * P.b_stride;
        bvar = P.bvar ? P.bvar + (size_t)lp * L : nullptr;
        bsign = P.bsign ? P.bsign + (size_t)lp * L : nullptr;
        brhs = P.brhs ? P.brhs + (size_t)lp * L : nullptr;
        ncols = n; nn = n - m;
        trace_out = (WARM && P.trace && lp == P.trace_lp) ? P.trace : nullptr;
        trace_cap = P.trace_cap;
        cur_phase = 2; cur_bland = 0;
    }
};

// Persistent CTA: pulls LP indices from a global counter until the batch is exhausted.
template <bool REG, bool WARM = true>
GM_DEV void cta_main(const BatchParams& P, double* wbase, double* bibase, double* small,
                     int* slot /* CTA-shared int */, double* ring = nullptr, unsigned long long* bars = nullptr) {
    SolverT<REG, WARM> s;
    s.bind_workspace(P, wbase, bibase, small, ring, bars);
    if (ring != nullptr) {
        if (gm_tid() == 0) {
            for (int k = 0; k < P.ring_stages; ++k) gm_mbar_init(bars + k, 1);
            gm_mbar_fence_init();
        }
        gm_sync();
    }
    for (;;) {
        if (gm_tid() == 0) {
            int it = gm_atomic_add(P.queue, 1);
            // streamed batches: the inputs of LP `it` may still be crossing PCIe; wait for the copy stream's counter
            if (P.ready != nullptr && it < P.count && !gm_wait_ready(P.ready, it)) it = -1 - it;
            *slot = it;
        }
        gm_sync();
        const int item = *slot;
        gm_sync();
        if (item >= P.count) break;
        if (item < 0) {  // the data never arrived (bounded wait): report, never hang
            if (gm_tid() == 0) P.status[-1 - item] = GM_ERR_CUDA;
            continue;
        }
        const int lp = P.lp_list ? P.lp_list[item] : item;
        s.bind_lp(P, lp);
        s.solve(P, lp);
    }
}

// Cooperative tier: CTA b is rank b % G of group b / G. The leader pulls LPs from the queue and solves them with the
// group's help; the helpers serve until the leader posts CMD_EXIT. `smem` = this CTA's dynamic shared memory.
GM_DEV void coop_cta_main(const BatchParams& P, double* smem, int* slot) {
    SolverT<false, true, true> s;
    const int G = P.coop_G, T = gm_nthreads();
    const int grp = gm_block_id() / G;
    const int m = P.m0 + P.L, n = P.n0 + P.L;
    const WsLayout w = ws_layout(m, n, T, false, true);
    const CoopLayout c = coop_layout(m, n, T, G, P.coop_pan == 16 ? (size_t)1 << 30 : 0);
    double* base = P.work + (size_t)grp * P.work_stride;
    // the host decided (BatchParams::coop_small) whether the vectors fit in shared memory beside the scratch
    double* small = P.coop_small ? smem + c.s_small : base + w.big_doubles;
    s.bind_workspace(P, base + w.W, base + w.Bi, small, nullptr, nullptr);
    s.G = G;
    s.rank = gm_block_id() % G;
    s.gbar = P.coop_bar + grp;
    s.epoch = 0;
    s.mail = base + c.mail;
    s.Bi1 = base + c.Bi1; s.Tp = base + c.Tp; s.Rs = base + c.Rs;
    s.s_y = smem + c.s_y; s.s_prow = smem + c.s_prow; s.s_ae = smem + c.s_ae; s.s_xb = smem + c.s_xb;
    s.s_al = smem + c.s_al; s.s_f = smem + c.s_f; s.s_r = smem + c.s_r; s.s_part = smem + c.s_part;
    s.s_pan = P.coop_pan == 16 ? smem : nullptr;             // aliases the scratch above (see coop_layout)
    for (int k = 0; k < 8; ++k) s.prof_t[k] = 0;
    s.red = smem + c.s_red;                                   // block reductions go through shared memory
    s.s_bit = reinterpret_cast<int*>(smem + c.s_bit);
    s.redi = reinterpret_cast<int*>(smem + c.s_redi);
    if (s.rank != 0) {
        s.piv1 = s.piv2 = s.ninv = 0;
        s.trace_out = nullptr;
        s.coop_helper_loop();
        return;
    }
    for (;;) {
        if (gm_tid() == 0) {
            int it = gm_atomic_add(P.queue, 1);
            if (P.ready != nullptr && it < P.count && !gm_wait_ready(P.ready, it)) it = -1 - it;
            *slot = it;
        }
        gm_sync();
        const int item = *slot;
        gm_sync();
        if (item >= P.count) break;
        if (item < 0) {
            if (gm_tid() == 0) P.status[-1 - item] = GM_ERR_CUDA;
            continue;
        }
        const int lp = P.lp_list ? P.lp_list[item] : item;
        s.bind_lp(P, lp);
        for (int k = 0; k < 16; ++k) s.prof_t[k] = 0;
        const long long t0 = gm_clock();
        s.solve(P, lp);
        s.prof_add(0, t0);
        if (P.prof && gm_tid() == 0)
            for (int k = 0; k < 16; ++k) P.prof[(size_t)lp * 16 + k] = s.prof_t[k];
    }
    s.coop_post_exit();
}

}  // namespace gm
