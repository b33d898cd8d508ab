/* gomilp_b200.h — C ABI of libgomilp_b200.so, the B200 LP-relaxation engine behind GoMILP.
 *
 * Every entry point is what a cgo binding on the reference side would call (INTEGRATION.md shows the
 * stubs). Plain pointers and sizes only; caller owns every buffer; nothing is retained after return
 * (the cgo pointer rule), so host-buffer entry points copy synchronously. There is NO CPU fallback:
 * without a CUDA device every compute call returns GM_ERR_NO_DEVICE.
 *
 * Reference interfaces replaced (paths relative to /root/reference):
 *   gm_simplex            lp.Simplex(c, A, b, tol, initialBasic)
 *                         vendor/gonum.org/v1/gonum/optimize/convex/lp/simplex.go:88-91
 *   gm_simplex_batch*     the same call made `count` times by solveWorker goroutines, tree.go:196-205
 *   gm_upload_root        milpProblem.toInitialSubproblem, ilp.go:43-71 (the shared c, A, b every node points to)
 *   gm_solve_wave         subProblem.solve for a whole FIFO wave of nodes, subproblem.go:141-187
 *                         (combineInequalities :55-78 + convertToEqualities :81-139 + lp.Simplex :154)
 *   gm_milp_solve         milpProblem.solve, ilp.go:75-116 -> enumerationTree.startSearch, tree.go:66-123
 *   gm_last_timing        extension of the BnbMiddleware hook, instrumentation.go:8-15 (per-wave device timings)
 */
#ifndef GOMILP_B200_H
#define GOMILP_B200_H

#include <stdint.h>

#include "gomilp_status.h"

#ifdef __cplusplus
extern "C" {
#endif

/* ---- lifecycle ------------------------------------------------------------------------------- */
int gm_device_count(void);       /* number of CUDA devices visible, 0 if none */
int gm_init(int device);         /* bind the CALLING THREAD to `device` (one engine context per device; threads that
                                    never call gm_init use the first device initialised); GM_OK / GM_ERR_NO_DEVICE /
                                    GM_ERR_CUDA. Roots remember their device: a wave runs where its root lives. */
int gm_shutdown(void);           /* release roots, streams and cached workspaces */
const char* gm_last_error(void); /* message of the last GM_ERR_CUDA on the calling thread */

/* Device timings of the last compute call made by the calling thread. */
typedef struct gm_timing {
    double h2d_ms;      /* host -> device copies */
    double kernel_ms;   /* simplex kernel(s), CUDA events on the launch stream */
    double d2h_ms;      /* device -> host copies */
    int64_t lps;        /* LP relaxations solved */
    int64_t launches;   /* kernel launches */
    int64_t smem_bytes; /* dynamic shared memory per CTA (0: HBM-resident tier) */
    int32_t tier;       /* 1 = basis inverse in registers + W in shared memory (m <= 64), 2 = all in shared memory,
                           3 = inverse + vectors in shared memory, W in HBM, 4 = W and inverse in HBM behind a TMA
                           staging ring, vectors in shared memory, 5 = all in HBM, 6 = cooperative: several CTAs
                           (grid / LPs) share one LP, state in HBM / L2 (fewer LPs than SMs) */
    int32_t grid, block;
} gm_timing;
int gm_last_timing(gm_timing* out);

/* Engine knobs with reference-compatible defaults (0 / negative = default). */
typedef struct gm_options {
    int32_t max_pivots;      /* safety cap per LP; the reference has none. default 50*(m+n)+1000. A cap set here bounds
                                the pivots of all passes of an LP together, robust passes included: an LP that reaches
                                it returns GM_ERR_ITERATION_LIMIT. Only the default cap is raised by the robust passes. */
    int32_t refactor_period; /* pivots between rebuilds of the basis inverse. default 100 */
    int32_t force_tier;      /* 0 auto, else the gm_timing.tier to force (GM_ERR_TOO_LARGE if it does not fit) */
    int32_t reserved;        /* 1: tier 4 without the TMA staging ring (plain loads), for A/B measurements */
    int32_t coop_group;      /* tier 6: CTAs per LP. default min(SMs / LPs in the launch, m / 2) */
    int32_t reserved2;       /* 1: large pinned host batches use one launch per slice instead of one launch gated on
                                arrival counters (A/B measurements) */
    int32_t robust;          /* 1: NOT the reference's behaviour. An LP on which the reference's rule set gives up
                                (ErrBland, mat.Condition after zero-step pivots, the pivot cap where the reference would
                                cycle) is solved once more on a right-hand side perturbed by ~1e-7 relative and the basis
                                found re-evaluated on the true one; stats[5] bit 1 marks such LPs. Default 0: the failure
                                is reported like the reference's error value. */
    int32_t reserved3;
} gm_options;
int gm_set_options(const gm_options* opt); /* process-wide */
/* Per-thread robust depth: while > 0, every wave the calling thread launches solves with gm_options.robust = 1
 * whatever the process-wide options say (gm_milp_solve uses it for GM_BNB_ROBUST). Returns the new depth. */
int gm_thread_robust(int delta);

/* Cooperative tier (6) only: arm before a host-buffer compute call; every LP of that call reports 16 int64: SM clock
 * cycles its leader CTA spent in [0] the whole solve, [1] the cooperative main loop, [2] basis inversions, [3] polish
 * (refinement, may nest an inversion), [4] leader-only Bland pivots, [5] periodic refactorisation, and the counts
 * [6] main-loop entries, [7] polish calls; cycles in [8] the input checks, [9] the warm start, [10] initial basis / Phase-I
 * set-up, [11] the Phase-I repair loop, [12] writing results, [13] main-loop entry / exit; [14..15] reserved.
 * The per-wave device-timing extension of BnbMiddleware, one level down. */
int gm_profile_arm(void);
int64_t gm_profile_fetch(int64_t* out /* [lps][16] */, int64_t lps);

/* Measured shared-memory bandwidth of the current device in GB/s (all SMs streaming conflict-free 16-byte loads):
 * the denominator of the roofline of the shared-memory resident tiers (bench.py). */
int gm_microbench_smem_gbs(double* gbs_out);

/* Pivot trace (parity evidence, BASELINE.json "identical ... branching sequences where pivots tie-break
 * identically"): arm before a host-buffer compute call on this thread; LP `lp_index` of that call records its first
 * `cap` pivots as int32 rows (phase 1|2, entering variable, leaving variable, chosen by replaceBland 0|1) - the
 * quantities simplex.go:233-293 decides per iteration. gm_trace_fetch copies up to cap rows (-1 = unused). */
int gm_trace_arm(int64_t lp_index, int64_t cap);
int64_t gm_trace_fetch(int32_t* rows, int64_t cap);

/* ---- (1) one LP: lp.Simplex, simplex.go:88 -----------------------------------------------------
 * min c'x s.t. Ax = b, x >= 0. A row-major m x n with row stride lda (mat.Dense layout).
 * initialBasic: NULL or m column indices of a feasible basis (simplex.go:147-160; an infeasible or
 * singular one returns GM_PANIC_INITIAL_BASIC where the reference panics).
 * Returns the gm_status. optF: objective (-Inf when unbounded, NaN when the reference returns NaN).
 * optX (n): solution, zeros when the reference returns nil. basisOut (m, may be NULL). pivots (may be NULL). */
int gm_simplex(const double* c, const double* A, int64_t lda, const double* b, int64_t m, int64_t n, double tol,
               const int64_t* initialBasic, double* optF, double* optX, int64_t* basisOut, int64_t* pivots);

/* ---- (1b) `count` independent LPs of one shape, HOST buffers ------------------------------------
 * c [count][n], A [count][m][n], b [count][m]; status [count], optF [count], optX [count][n],
 * basis [count][m] (may be NULL), stats [count][8] (may be NULL: pivots phase I, phase II, Bland calls,
 * basis inversions, used phase I, basis-scan fallback, repair trials, x non-nil).
 * Returns GM_OK when the batch ran (per-LP outcomes are in status[]), else an engine code. */
int gm_simplex_batch(int64_t count, const double* c, const double* A, const double* b, int64_t m, int64_t n,
                     double tol, int32_t* status, double* optF, double* optX, int64_t* basis, int32_t* stats);

/* ---- (1c) same, DEVICE buffers, asynchronous on `stream` (a cudaStream_t; NULL = default stream) --- */
int gm_simplex_batch_device(int64_t count, const double* d_c, const double* d_A, const double* d_b, int64_t m,
                            int64_t n, double tol, int32_t* d_status, double* d_optF, double* d_optX,
                            int64_t* d_basis, int32_t* d_stats, void* stream);

/* ---- (2) frontier wave over one shared root ---------------------------------------------------- */
typedef int64_t gm_root_t;
/* Upload the root standard form (c0 [n0], A0 [m0][lda], b0 [m0]) once; every node of every wave reads it. */
int gm_upload_root(const double* c0, const double* A0, int64_t lda, const double* b0, int64_t m0, int64_t n0,
                   gm_root_t* out);
int gm_free_root(gm_root_t root);
/* Solve `nodes` sub-problems of depth L in one launch. Node k carries L branch rows
 * (bvar[k][l], bsign[k][l], brhs[k][l]) = bnbConstraint{branchedVariable, gsharp[var], hsharp}
 * (subproblem.go:36-44); its LP is [A0 0; G I] x = [b0; h] of shape (m0+L) x (n0+L).
 * Outputs: status [nodes], z [nodes], x [nodes][n0] (truncated like subproblem.go:157-159),
 * basis [nodes][m0+L] (may be NULL), stats [nodes][8] (may be NULL). */
int gm_solve_wave(gm_root_t root, int64_t nodes, int64_t L, const int32_t* bvar, const double* bsign,
                  const double* brhs, int32_t* status, double* z, double* x, int64_t* basis, int32_t* stats);

/* Warm-started wave (north star: "children warm-start from the parent basis"). Same as gm_solve_wave, plus
 * parent[k] = index of node k's parent in the PREVIOUS gm_solve_wave_warm call on this root (which must have had
 * depth L-1), or -1 for a cold start; parent == NULL = all cold. The engine keeps every node's final basis and
 * basis inverse of the last warm wave in HBM (nodes x (m^2 + m) x 8 B; skipped when it would not fit), and a child
 * starts from [B 0; g 1]^-1 = [B^-1 0; -g B^-1 1] without any factorisation. Optimal objective and x are those of
 * the cold solve whenever the optimum is unique; the pivot path differs, so this is not a replay of lp.Simplex's
 * initialBasic = nil call (subproblem.go:154) and is off by default in gm_milp_solve. */
int gm_solve_wave_warm(gm_root_t root, int64_t nodes, int64_t L, const int32_t* bvar, const double* bsign,
                       const double* brhs, const int32_t* parent, int32_t* status, double* z, double* x,
                       int64_t* basis, int32_t* stats);

/* ---- (3) whole MILP: milpProblem.solve, ilp.go:75-116 ------------------------------------------- */
typedef struct gm_milp_result {
    int32_t status;     /* gm_milp_status */
    int32_t lp_status;  /* offending gm_status for the PANIC_* outcomes */
    double z;
    int64_t x_len;      /* entries written to x (nvar, or nvar+nineq on a deadline: ilp.go:92-99 does not strip slacks) */
    int64_t nodes;      /* LP relaxations solved, root included */
    int64_t waves;      /* kernel launches = BFS levels processed */
    int64_t pivots;
    double device_ms;   /* sum of kernel times */
} gm_milp_result;

/* Per-node decision callback = BnbMiddleware.ProcessDecision (instrumentation.go:8-15), invoked in the
 * 1-worker FIFO order of the reference; NewSubProblem is implied by (id, parent). May be NULL. */
typedef void (*gm_decision_cb)(void* user, int64_t id, int64_t parent, int32_t depth, int32_t lp_status, double z,
                               int32_t decision, int32_t branch_var, double branch_floor);
/* Per-wave callback (the device-timing extension). May be NULL. */
typedef void (*gm_wave_cb)(void* user, int64_t wave, int64_t nodes, int64_t pivots, double kernel_ms);

/* c [nvar]; A [meq][nvar], b [meq] (meq may be 0); G [nineq][nvar], h [nineq] (nineq may be 0);
 * integrality [nvar] (0/1). heuristic: gm_branch_heuristic; mode: gm_bnb_mode, optionally | GM_BNB_WARM_START.
 * node_limit / time_limit_s stand in for the context deadline (0 = none).
 * x must hold nvar + nineq + 1 doubles. */
int gm_milp_solve(int64_t nvar, const double* c, int64_t meq, const double* A, const double* b, int64_t nineq,
                  const double* G, const double* h, const uint8_t* integrality, int32_t heuristic, int32_t mode,
                  int64_t node_limit, double time_limit_s, double* x, gm_milp_result* result,
                  gm_decision_cb on_decision, gm_wave_cb on_wave, void* user);

/* ---- (3b) the same search with the decisions made on the device, optionally sharded over several GPUs ------------
 * gm_milp_solve_device = gm_milp_solve(..., mode | GM_BNB_DEVICE_SCAN, ...): tree.go's FIFO queue becomes a per-GPU
 * wavefront, checkSolution (tree.go:207-263) an exclusive prefix-min scan over 32-byte node records, branching.go
 * reads x from device buffers. With a communicator (below) every rank calls it with IDENTICAL arguments: rank r solves
 * the r-th contiguous FIFO block of every wave, the node records are exchanged with one ncclAllGather per wave over
 * NVLink, and every rank returns the same result (the incumbent's x is broadcast from the rank that found it).
 * time_limit_s is honoured only without a communicator (ranks must agree on where to stop: use node_limit). */
int gm_milp_solve_device(int64_t nvar, const double* c, int64_t meq, const double* A, const double* b, int64_t nineq,
                         const double* G, const double* h, const uint8_t* integrality, int32_t heuristic, int32_t mode,
                         int64_t node_limit, double time_limit_s, double* x, gm_milp_result* result,
                         gm_decision_cb on_decision, gm_wave_cb on_wave, void* user);

/* Communicator of the calling thread (one rank per GPU; NCCL is loaded at run time, libnccl.so.2).
 * Rank 0 creates the 128-byte id and hands it to the other ranks by any means (the Go side: a channel or a file;
 * the tests: torch.distributed / multiprocessing). gm_comm_init binds the rank to the thread's current device. */
int gm_comm_unique_id(void* id128);
int gm_comm_init(int32_t rank, int32_t world, const void* id128);
int gm_comm_destroy(void);

#ifdef __cplusplus
}
#endif
#endif /* GOMILP_B200_H */
