/*
 * lfr.h — C ABI of the multi-view local-feature refinement solve.
 *
 * This is the drop-in boundary for the hot path of
 * mihaidusmanu/local-feature-refinement, multi-view-refinement/solve.cc.
 * The reference has no in-process boundary: it solves every component on a
 * thread pool by calling
 *
 *     create_and_solve_problem(graph, track_idx, positions, is_root,
 *                              component_idx, nodes_in_component, 1)
 *                                                     (solve.cc:79-87, :617-635)
 *
 * lfr_solve() replaces that whole dispatch loop (solve.cc:614-635) in one
 * call; the arrays in lfr_problem are exactly the arguments of
 * create_and_solve_problem in structure-of-arrays form.
 *
 * Two libraries export this same header:
 *   liblfr_b200.so — the product: hand-written sm_100a CUDA, no CPU fallback.
 *   liblfr_ref.so  — the CPU oracle (oracle/), test infrastructure only.
 *
 * Conventions: plain pointers and sizes; the caller owns every buffer and the
 * library never retains one after a call returns (plans copy what they need);
 * functions return 0 or a negative LFR_E* code and never throw or abort
 * across the ABI; lfr_last_error() is thread-local.
 */
#ifndef LFR_H_
#define LFR_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LFR_ABI_VERSION 1

/* ---- error codes ------------------------------------------------------- */
#define LFR_OK 0
#define LFR_EINVAL (-1)    /* malformed problem / NULL pointer                */
#define LFR_ENODEV (-2)    /* no CUDA device / CUDA extension unusable        */
#define LFR_ECUDA (-3)     /* a CUDA runtime call failed                      */
#define LFR_ENOMEM (-4)
#define LFR_EUNSUPPORTED (-5)

/* ---- per-edge loss kinds (solve.cc:105-125) ---------------------------- */
#define LFR_EDGE_SKIP 0   /* other component: no residual block (solve.cc:123) */
#define LFR_EDGE_CAUCHY 1 /* same track:  sim * CauchyLoss(0.25)  (solve.cc:111) */
#define LFR_EDGE_TUKEY 2  /* same component, other track: sim * TukeyLoss(0.0625) (solve.cc:120) */

/* ---- termination codes (Ceres TrustRegionMinimizer, SURVEY Appendix A.6) */
#define LFR_TERM_SKIPPED 0        /* component of size 1 (solve.cc:619-622)   */
#define LFR_TERM_GRADIENT_TOL 1   /* max-norm of projected gradient <= 1e-8   */
#define LFR_TERM_PARAMETER_TOL 2  /* |step| <= 1e-4 (|x| + 1e-4)              */
#define LFR_TERM_FUNCTION_TOL 3   /* |dcost| <= 1e-4 cost                     */
#define LFR_TERM_MIN_RADIUS 4     /* trust region radius <= 1e-32             */
#define LFR_TERM_NO_CONVERGENCE 5 /* 100 iterations                           */
#define LFR_TERM_FAILURE 6        /* 10 consecutive invalid steps             */
#define LFR_TERM_EMPTY 7          /* no non-constant parameter block          */

/*
 * One directed edge of the match graph (graph.h:11-19), as laid out in HBM:
 * 80 bytes, 16-byte aligned => five 128-bit loads.  The flow grid stays fp32
 * (it is `float` on the wire, types.proto:16-17) and is widened to fp64 in
 * registers, which is bit-identical to the reference's vector<double> copy
 * (solve.cc:460-472).
 *   flow[2*(3*i+j)+k] : 3x3 grid, i = row sample, j = col sample in
 *                       {-0.5, 0, +0.5}; k = 0 -> di (row), 1 -> dj (col)
 *                       (cost.cc:34, solve.cc:461-464)
 */
typedef struct lfr_edge {
  float flow[18];
  float sim;    /* similarity = ScaledLoss weight (solve.cc:111,120) */
  uint32_t dst; /* destination node index (graph.h:15)                */
} lfr_edge;

/*
 * The problem: the reference's Graph (out-edge lists, graph.h:21-41) as CSR by
 * source node, plus the per-node containers of solve.cc.
 */
typedef struct lfr_problem {
  uint32_t n_nodes;
  uint32_t n_components;  /* entries in comp_ptr - 1                         */
  uint64_t n_edges;       /* directed edges = row_ptr[n_nodes]               */
  const uint32_t* row_ptr;   /* [n_nodes+1]  out-edges of node v: edges[row_ptr[v] .. row_ptr[v+1]) in insertion order */
  const lfr_edge* edges;     /* [n_edges]                                    */
  const uint32_t* track;     /* [n_nodes]  track_idx_container (solve.cc:526-541) */
  const uint32_t* comp;      /* [n_nodes]  component_idx_container (solve.cc:586) */
  const uint8_t* is_root;    /* [n_nodes]  is_root (solve.cc:570-582)        */
  const uint32_t* comp_ptr;  /* [n_components+1]  dispatch list, largest first (solve.cc:599-604) */
  const uint32_t* comp_nodes;/* [comp_ptr[n_components]] nodes_in_component, ascending node index (solve.cc:594-597) */
} lfr_problem;

/* Every constant of solve.cc:89,111,120,146-154 and the Ceres defaults in
 * force (SURVEY Appendix A.5).  lfr_options_default() fills the reference's
 * values. */
typedef struct lfr_options {
  double bound;                   /* 1.0      solve.cc:89                   */
  double cauchy_a;                /* 0.25     solve.cc:111                  */
  double tukey_a;                 /* 0.0625   solve.cc:120                  */
  int32_t tukey_variant;          /* 1 = Ceres 1.x (a^2/6), 2 = Ceres 2.x (a^2/3) */
  int32_t max_num_iterations;     /* 100      solve.cc:149                  */
  int32_t max_num_consecutive_invalid_steps; /* 10  solve.cc:151            */
  int32_t max_num_line_search_step_size_iterations; /* 20                   */
  double function_tolerance;      /* 1e-4     solve.cc:152                  */
  double gradient_tolerance;      /* 1e-8     solve.cc:153                  */
  double parameter_tolerance;     /* 1e-4     solve.cc:154                  */
  double initial_trust_region_radius; /* 1e4                                */
  double max_trust_region_radius;     /* 1e16                               */
  double min_trust_region_radius;     /* 1e-32                              */
  double min_relative_decrease;       /* 1e-3                               */
  double min_lm_diagonal;             /* 1e-6                               */
  double max_lm_diagonal;             /* 1e32                               */
  double line_search_sufficient_function_decrease; /* 1e-4                  */
  double max_line_search_step_contraction;         /* 1e-3                  */
  double min_line_search_step_contraction;         /* 0.6                   */
  double min_line_search_step_size;                /* 1e-9                  */
  int32_t n_threads;     /* CPU oracle: pool threads (solve.cc:384,617). b200: ignored */
  int32_t device;        /* b200: CUDA device ordinal; oracle: ignored      */
  int32_t linear_solver; /* 0 auto, 1 dense Cholesky, 2 block-Jacobi PCG (b200 only) */
  int32_t debug_flags;   /* LFR_DBG_* test / profiling hooks; 0 in production      */
} lfr_options;

/* lfr_options.debug_flags (b200 only): route components through the fallback tiers, switch the
 * zero-copy mechanism off, collect per-component cycle counters.  Results do not depend on them
 * (tests/test_gpu_parity.py).  Other bits are ignored. */
#define LFR_DBG_FORCE_SMEM_CHOLESKY 0x1 /* every warp-tier component through the shared-memory Cholesky kernel */
#define LFR_DBG_NO_TILE 0x2             /* no 64/128-thread tile kernels                                       */
#define LFR_DBG_NO_ZERO_COPY 0x8        /* lfr_solve(): copy edges / positions through HBM even when the caller's buffers are pinned */
#define LFR_DBG_PROFILE 0x10            /* per-component clock64() counters (lfr_debug_plan_cycles)            */

/* Optional per-component results, caller-owned, indexed like comp_ptr. Any
 * pointer may be NULL. */
typedef struct lfr_stats {
  int32_t* iterations;    /* [n_components] LM iterations run (Ceres summary.iterations.size() - 1) */
  int32_t* termination;   /* [n_components] LFR_TERM_*                       */
  double* initial_cost;   /* [n_components] cost at iteration 0 (fixed root-root cost excluded, A.1) */
  double* final_cost;     /* [n_components] cost at the returned positions   */
  /* totals, filled by the library */
  uint64_t total_iterations;
  uint64_t total_line_search_steps;
  uint32_t n_solved;      /* components of size > 1                          */
  uint32_t n_kernel_launches; /* b200: kernels launched by this call         */
  double h2d_ms, kernel_ms, d2h_ms, total_ms; /* b200: CUDA-event timings; oracle: total_ms = pool wall time */
} lfr_stats;

int lfr_abi_version(void);
/* "b200" or "cpu-oracle" */
const char* lfr_backend(void);
const char* lfr_last_error(void);
void lfr_options_default(lfr_options* o);

/*
 * Solve every component of size > 1.  `positions` is [2*n_nodes] doubles,
 * (row, col) per node (cost.cc:83): in = initial values (the reference passes
 * zeros, solve.cc:609-612), out = refined displacements; entries of nodes that
 * are roots, or in components of size 1, are left untouched, and so is a
 * component whose solve ends in LFR_TERM_FAILURE (Ceres only commits a usable
 * solution).  Replaces solve.cc:614-635.  Host pointers; host<->device traffic
 * inside the call.  b200: when `p->edges` / `positions` are page-locked host
 * memory (cudaHostAlloc / cudaHostRegister, 16-byte aligned) the kernels pull
 * each component's edge records straight from the caller's buffer into shared
 * memory (zero-copy over PCIe, overlapped with the solves) and write the
 * results straight back; pageable buffers are copied through HBM.
 */
int lfr_solve(const lfr_problem* p, const lfr_options* o, double* positions,
              lfr_stats* stats);

/*
 * The same solve on several GPUs of one node from ONE call (SURVEY 8b / 8e: "one call drives
 * 1..8 GPUs").  Components are independent (solve.cc:123-125 drops cross-component edges,
 * solve.cc:586 caps a component at #images nodes), so the dispatch slots are LPT-packed over
 * `devices` by directed-edge count — the reference's largest-first queue (solve.cc:599-604) spread
 * over devices — and every device solves its slots concurrently.  With page-locked `p->edges` /
 * `positions` each device pulls only ITS components' edge records from the shared host array and
 * writes its results straight back (disjoint entries): the edge data is partitioned without being
 * copied or replicated and no collective is needed; the small per-node arrays are replicated.
 * Pageable buffers go through each device's HBM (edges replicated) and are merged on the host.
 * Results are bitwise identical to lfr_solve() on one device.  `info` may be NULL.
 * The oracle exports the symbol and ignores `devices`.
 */
typedef struct lfr_multi_info {
  double kernel_ms[16], total_ms[16];  /* per entry of `devices`                               */
  uint32_t n_slots[16];                /* components solved by that device                     */
  uint64_t n_edges[16];                /* their directed edges (the LPT weight)                */
  int32_t zero_copy, reserved;
} lfr_multi_info;

int lfr_solve_multi(const lfr_problem* p, const lfr_options* o, const int32_t* devices, int32_t n_devices,
                    double* positions, lfr_stats* stats, lfr_multi_info* info);

/* lfr_solve() / lfr_solve_multi() keep one grow-only workspace per device between calls (device
 * buffers, pinned staging, streams) so that steady-state calls allocate nothing.  lfr_shutdown()
 * releases them all; a later call simply re-creates what it needs.  No-op in the oracle. */
void lfr_shutdown(void);

/* Page-locked host memory for the arrays handed to lfr_solve() / lfr_solve_multi(): `edges` and
 * `positions` allocated here are used in place (zero-copy, see lfr_solve).  Returns NULL when the
 * allocation fails or there is no CUDA device — the caller may then use ordinary memory (the solve
 * still needs a device).  The oracle returns ordinary aligned memory.  Free with lfr_host_free(). */
void* lfr_host_alloc(uint64_t bytes);
void lfr_host_free(void* p);

/* ---- device-resident plan (b200 only; the oracle returns LFR_EUNSUPPORTED) --
 * lfr_plan_create copies the problem to HBM once; lfr_plan_solve re-runs the
 * whole solve from the stored initial positions, asynchronously on `stream`
 * (a cudaStream_t, NULL = the legacy default stream); lfr_plan_download
 * synchronises and copies positions / stats back. */
typedef struct lfr_plan lfr_plan;
int lfr_plan_create(const lfr_problem* p, const lfr_options* o,
                    const double* initial_positions /* [2N] or NULL = zeros */,
                    lfr_plan** out);
int lfr_plan_solve(lfr_plan* plan, void* stream);
int lfr_plan_download(lfr_plan* plan, void* stream, double* positions,
                      lfr_stats* stats);
/* number of kernels one lfr_plan_solve launches */
int lfr_plan_num_launches(const lfr_plan* plan);
/* algorithmic bytes of the last completed solve: sum_c iters_c*(80 E_c + 36 N_c)
 * and the one-pass lower bound 80 E + 36 N over solved components (SURVEY 8d) */
int lfr_plan_traffic(lfr_plan* plan, void* stream, uint64_t* algorithmic_bytes,
                     uint64_t* one_pass_bytes);
void lfr_plan_destroy(lfr_plan* plan);

/* ---- test hooks: per-edge evaluation (K1; cost.cc:13-48,78-90 + loss) -------
 * For edge e: x1 = xs[2e..], x2 = xd[2e..]; outputs residual r[2e..] (raw),
 * jac[4e..] = d r / d x1 row-major (raw, = -(I+G)), rho[3e..] = scaled loss
 * {rho, rho', rho''} at |r|^2.  kind[e] in LFR_EDGE_*. */
int lfr_debug_edge_eval(const lfr_edge* edges, const uint8_t* kind, uint64_t n,
                        const double* xs, const double* xd,
                        const lfr_options* o, double* r, double* jac,
                        double* rho);

#ifdef __cplusplus
}
#endif
#endif /* LFR_H_ */
