/* libppgpu - C ABI of the B200 engine for PPOPT's combinatorial mpQP/mpLP critical-region enumeration.
 *
 * The reference (TAMUparametric/PPOPT) is pure Python and has no FFI for this path; the seam it offers is the call
 *     mpqp_combinatorial.solve(program) -> Solution      (src/ppopt/mp_solvers/mpqp_combinatorial.py:10-72,
 *                                                         dispatched from src/ppopt/mp_solvers/solve_mpqp.py:70-71)
 * Each entry point below replaces the body of one piece of that function for a whole LEVEL of candidate active
 * sets at once.  All `d_` pointers are device pointers owned by the caller (the Python host passes
 * torch tensor data_ptr()s), all `h_` pointers are host pointers; nothing is retained after a call returns except
 * the opaque program handle.  Every function returns 0 on success and a negative code on failure, in which case
 * ppgpu_last_error() describes it.  A handle is not thread-safe; different handles may be used concurrently.
 *
 * Candidate active sets are bitmasks over the INEQUALITY rows of the main constraint body: bit i of word i/64
 * stands for constraint row n_eq + i (equality rows 0..n_eq-1 are always active, mplp_program.py:112-118).
 * A level's candidates are stored as n x words uint64, in the reference's lexicographic order.
 */
#ifndef PPGPU_H
#define PPGPU_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct ppgpu_program ppgpu_program;
typedef void* ppgpu_stream; /* cudaStream_t */

/* sizes of one program, after the reference's own presolve (program constructor) has run */
typedef struct {
    int32_t n;     /* num_x()            mplp_program.py:140-142 */
    int32_t t;     /* num_t()            mplp_program.py:144-146 */
    int32_t m;     /* num_constraints()  mplp_program.py:148-150 */
    int32_t q;     /* rows of A_t */
    int32_t n_eq;  /* len(equality_indices), equalities are rows 0..n_eq-1 */
    int32_t is_qp; /* 1: MPQP_Program (Q given), 0: MPLP_Program */
} ppgpu_dims;

typedef struct {
    int32_t words;        /* uint64 words per candidate bitmask */
    int32_t n_ineq;       /* m - n_eq */
    int32_t region_rows;  /* rows of the theta-space polytope before filtering: (m - n_eq) + q */
    int32_t use_gram;     /* 1: Cholesky/Schur optimality screen available (Q symmetric positive definite) */
    int32_t max_depth;    /* max(n, t) - n_eq   mpqp_combinatorial.py:24 */
    int32_t sm_count;
    int32_t lp_columns;   /* padded register columns of the feasibility tableau */
    int32_t reserved;     /* 1: the vertex walk (K2w) has a start vertex for this program */
} ppgpu_info;

/* number of uint64 counters returned by ppgpu_counters */
#define PPGPU_NUM_COUNTERS 27

const char* ppgpu_last_error(void);
int ppgpu_version(void);

/* Upload a program and precompute everything that is shared by all candidates (equality elimination, Gram matrix).
 * Arrays are row-major float64 host arrays with the shapes of the reference's attributes
 * (A m x n, b m, F m x t, A_t q x t, b_t q, Q n x n or NULL, c n, H n x t).  mplp_program.py:45-58 */
int ppgpu_program_create(const ppgpu_dims* dims, const double* h_A, const double* h_b, const double* h_F,
                         const double* h_A_t, const double* h_b_t, const double* h_Q, const double* h_c,
                         const double* h_H, int device, ppgpu_program** out);
int ppgpu_program_destroy(ppgpu_program* prog);
int ppgpu_program_info(const ppgpu_program* prog, ppgpu_info* out);

/* Engine knobs of one handle (no reference counterpart: the reference has one LP call per candidate and nothing to tune).
 *   PPGPU_OPT_K2W_MIN  smallest number of candidates per ppgpu_level_eval chunk for which the feasibility certificates are
 *                      produced by the vertex walk (csrc/k2w_walk.cu) before the relaxation (default 100000; 0: always;
 *                      negative: never).  Decisions do not depend on it - only which kernel exhibits the feasible point. */
#define PPGPU_OPT_K2W_MIN 0
/*   PPGPU_OPT_K2W_REF  1: the vertex walk applies every pivot to its whole dictionary (the reference of the deferred
 *                      updates it uses by default where the dictionary's shape allows; results are identical); 0: default */
#define PPGPU_OPT_K2W_REF 1
/*   PPGPU_OPT_K2W_INFEAS  1 (default): a drive of the vertex walk that ends at the optimum of a candidate's last row proves
 *                      the candidate infeasible when its bound clears the feasibility tolerance by PPG_WALK_INF_MARGIN, and
 *                      the relaxation and the simplex skip it; 0: the walk only ever certifies feasibility (the reference
 *                      the tests compare against; results are identical) */
#define PPGPU_OPT_K2W_INFEAS 2
int ppgpu_set_option(ppgpu_program* prog, int32_t option, int64_t value);

/* Level-1 candidates = generate_children_sets(equality_indices, m, murder_list) (solver_utils.py:154-166) plus the mpLP
 * cardinality filter (mpqp_combinatorial.py:40-42).  d_masks must hold n_ineq x words uint64. */
int ppgpu_root_level(ppgpu_program* prog, uint64_t* d_masks, int64_t* h_count, ppgpu_stream stream);

/* check_child_feasibility + check_optimality for n candidates of cardinality n_eq + k_act:
 * K1 rank screen (is_full_rank, constraint_utilities.py:222-236), K2 feasibility LP (mplp_program.py:411-444),
 * K3/K4 optimality + full-dimension screen (mpqp_program.py:203-322, mpqp_utils.py:323-344).
 * Writes one status byte per candidate (PPG_ST_* bits of csrc/tolerances.h).  stages: bit0 K1, bit1 K2 (preceded by the
 * K2a relaxation certificates unless bit3 is set), bit2 K3/K4.  Asynchronous on `stream`; large n is processed in chunks
 * internally (PPGPU_CHUNK candidates), the library owns the K2a -> K2 hand-over scratch (grown on demand, pooled across
 * handles); d_masks / d_status may be arbitrary sub-ranges of a level (that is how a level is sharded between GPUs). */
int ppgpu_level_eval(ppgpu_program* prog, const uint64_t* d_masks, int64_t n, int32_t k_act, uint8_t* d_status,
                     int32_t stages, ppgpu_stream stream);

/* ppgpu_level_eval with feasibility WITNESSES (no reference counterpart: the reference solves one LP per candidate,
 * mplp_program.py:411-444, and shares nothing between candidates or levels).
 *   d_witness      (n x PPGPU_WITNESS_SLOTS x words uint64, zero-initialised by the caller, or NULL) receives, for every
 *                  candidate certified by the vertex walk or by inheritance, the mask of ALL rows active at the certifying
 *                  vertex (slot 0) and at a later vertex of the walk that holds the candidate too (slot 1, may stay 0);
 *   d_parent_*     (or NULL / 0) describe the level the candidates were generated from: the feasible masks and the
 *                  workspace exactly as ppgpu_children_count / ppgpu_children_prepare left them (the workspace holds the
 *                  prefix-group index of those masks), and the witnesses of those parents in the same order.  A candidate one of
 *                  whose parents has a witness that also holds the added row is certified by that same vertex before any
 *                  LP work is spent on it (and passes the witness on).
 * Decisions are identical with and without witnesses; only which kernel exhibits the feasible point changes. */
#define PPGPU_WITNESS_SLOTS 2
int ppgpu_level_eval_w(ppgpu_program* prog, const uint64_t* d_masks, int64_t n, int32_t k_act, uint8_t* d_status,
                       int32_t stages, uint64_t* d_witness, const uint64_t* d_parent_feas, int64_t parent_nf,
                       const void* d_parent_ws, const uint64_t* d_parent_wit, ppgpu_stream stream);

/* Workspaces.  K6 (ppgpu_children_*, n = nf): the scan scratch and the prefix-group index of the feasible parents
 * (~56 bytes per parent: a table, and per group the index of its first member and the bitmap of its members' highest
 * rows).  Ordered compaction (ppgpu_level_select): ~8 bytes per candidate; any workspace of
 * ppgpu_scan_workspace_bytes(n) bytes serves it as well. */
size_t ppgpu_scan_workspace_bytes(int64_t n);
size_t ppgpu_select_workspace_bytes(int64_t n);
/* Ordered compaction: ascending indices i with (d_status[i] & bits) == value.  Synchronises the stream to return the
 * count.  d_ws must hold ppgpu_select_workspace_bytes(n) bytes. */
int ppgpu_level_select(ppgpu_program* prog, const uint8_t* d_status, int64_t n, uint8_t bits, uint8_t value,
                       int64_t* d_idx_out, int64_t* h_count, void* d_ws, size_t ws_bytes, ppgpu_stream stream);

/* gen_cr_from_active_set (mpqp_utils.py:89-301) for the selected candidates d_sel[0..n_sel):
 *   d_laws  n_sel x (n + n_eq + k_act) x (t + 1)   [const | theta]: x-law rows then lambda-law rows
 *   d_rows  n_sel x region_rows x (t + 1)          [f | a] L2-normalised, reference row order
 *   d_flags n_sel x region_rows int32              bit0 nonzero row, bit1 non-redundant, bit2 duplicate
 *   d_info  n_sel x 4 float64                      {1 region / 0 none / -1 singular KKT, radius, lower, upper}
 * and sets PPG_ST_REGION in d_status for emitted regions. */
int ppgpu_regions_emit(ppgpu_program* prog, const uint64_t* d_masks, const int64_t* d_sel, int64_t n_sel,
                       int32_t k_act, double* d_laws, double* d_rows, int32_t* d_flags, double* d_info,
                       uint8_t* d_status, ppgpu_stream stream);

/* generate_children_sets + CombinationTester.check for all feasible parents (solver_utils.py:29-55,154-166):
 * pass 1 gathers the parents (d_feas_masks, nf x words), finds the surviving children of each (d_survive, nf x words)
 * and the exclusive scan of their counts (d_offsets, nf + 1); returns the total.  Pass 2 writes them, in order.
 * d_feas_idx selects the parents in the level's order, which is lexicographic (ppgpu_root_level, then this pass); a
 * selection that is not strictly increasing in that order, or mixes cardinalities, is an error (reported by this call
 * and by ppgpu_children_scan).  d_ws (ppgpu_scan_workspace_bytes(nf) bytes) keeps their prefix-group index for the
 * next level's ppgpu_level_eval_w. */
int ppgpu_children_count(ppgpu_program* prog, const uint64_t* d_masks, const int64_t* d_feas_idx, int64_t nf,
                         int32_t k_act, uint64_t* d_feas_masks, uint64_t* d_survive, int64_t* d_offsets,
                         int64_t* h_total, void* d_ws, size_t ws_bytes, ppgpu_stream stream);
/* The same pass 1 in three steps, for callers that split the parents between GPUs (SURVEY.md 8e): prepare gathers the
 * parents and builds their prefix-group index; count_range fills d_survive / d_counts for the parents [p_lo, p_hi) only (the
 * caller zero-fills both and sums them across ranks); scan turns the counts (nf + 1 entries) into offsets. */
int ppgpu_children_prepare(ppgpu_program* prog, const uint64_t* d_masks, const int64_t* d_feas_idx, int64_t nf,
                           uint64_t* d_feas_masks, void* d_ws, size_t ws_bytes, ppgpu_stream stream);
int ppgpu_children_count_range(ppgpu_program* prog, const uint64_t* d_feas_masks, int64_t nf, int32_t k_act,
                               uint64_t* d_survive, int64_t* d_counts, int64_t p_lo, int64_t p_hi, void* d_ws,
                               size_t ws_bytes, ppgpu_stream stream);
int ppgpu_children_scan(ppgpu_program* prog, int64_t* d_counts_to_offsets, int64_t nf, int64_t* h_total, void* d_ws,
                        size_t ws_bytes, ppgpu_stream stream);
int ppgpu_children_write(ppgpu_program* prog, const uint64_t* d_feas_masks, const uint64_t* d_survive,
                         const int64_t* d_offsets, int64_t nf, uint64_t* d_children, ppgpu_stream stream);

/* Batched point location + law evaluation for a solved program (Solution.get_region / evaluate, solution.py:44-112 with
 * region.is_inside, critical_region.py:81-84;  upop.PointLocation.locate / evaluate, upop/point_location.py:43-133).
 * Stateless - no program handle.
 *   d_theta   n_points x t                    parameter points
 *   d_rows    total_rows x (t + 1)            stacked half-spaces [f | E] of all regions, solution order
 *   d_row_off n_regions + 1                   first row of every region
 *   d_laws    n_regions x n_x x (t + 1)       [b | A] of every region (may be NULL when d_x is NULL and overlap is 0)
 *   use_tol   1: inside iff all(E theta - f < tol)   (Solution, tol = point_location_tolerance)
 *             0: inside iff all(E theta <= f)        (upop.PointLocation)
 *   overlap   0: the FIRST containing region (get_region_no_overlap)
 *             1: the containing region with the lowest objective 1/2 x'Qx + theta'H'x + c'x, ties to the later one
 *                (get_region_overlap); needs d_H (n_x x t), d_c (n_x) and, for an mpQP, d_Q (n_x x n_x, else NULL)
 *   d_region  n_points int32                  index of that region, -1 if none
 *   d_x       n_points x n_x or NULL          A theta + b of that region, NaN where d_region is -1 */
int ppgpu_locate_points(const double* d_theta, int64_t n_points, int32_t t, const double* d_rows, const int64_t* d_row_off,
                        int64_t n_regions, const double* d_laws, int32_t n_x, int32_t use_tol, double tol, int32_t overlap,
                        const double* d_Q, const double* d_H, const double* d_c, int32_t* d_region, double* d_x,
                        ppgpu_stream stream);

/* Batched fixed-parameter QP solves of an mpQP handle (MPQP_Program.solve_theta, mpqp_program.py, with the solver the
 * reference hands it to - daqp / gurobi / ... - and sample_theta_space; Solution.verify_solution's per-point QP solves).
 * A dual active-set iteration on the Gram data of the handle (csrc/k8_theta_qp.cu), one point per warp.
 *   d_theta   n_points x t          parameter points (the Theta rows A_t theta <= b_t do not constrain x: not imposed)
 *   d_status  n_points uint8        PPG_QP_* of csrc/tolerances.h: 0 optimal, 1 infeasible, 2 iteration cap, 3 numerical breakdown
 *   d_x       n_points x n or NULL  optimal x (NaN unless optimal)
 *   d_dual    n_points x m or NULL  multipliers of the rows: equality rows first (mu), then the inequality rows (lambda >= 0), so
 *                                   that Q x + H theta + c + A' dual = 0 (the convention of the regions' C theta + d laws)
 *   d_active  n_points x words or NULL  final working set, as a candidate mask (inequality rows only)
 *   d_iters   n_points int32 or NULL    steps taken (constraint additions + drops)
 * Asynchronous on `stream`.  Returns -2 for an mpLP handle or when use_gram is 0 (Hessian not positive definite on the space
 * left by the equalities). */
int ppgpu_solve_theta_batch(ppgpu_program* prog, const double* d_theta, int64_t n_points, uint8_t* d_status, double* d_x,
                            double* d_dual, uint64_t* d_active, int32_t* d_iters, ppgpu_stream stream);

/* Batched fixed-parameter LP solves of an mpLP handle (MPLP_Program.solve_theta, mplp_program.py, with the LP backend the
 * reference hands it to - GLPK / HiGHS / ... - and sample_theta_space; Solution.verify_solution's per-point LP solves).
 * A dense primal dictionary simplex (Phase 1 with one auxiliary column, then Phase 2) from the theta-independent start
 * dictionary of the handle (csrc/k9_theta_lp.cu), one point per warp.
 *   d_theta   n_points x t          parameter points (the Theta rows A_t theta <= b_t do not constrain x: not imposed)
 *   d_status  n_points uint8        PPG_TLP_* of csrc/tolerances.h: 0 optimal, 1 infeasible, 2 iteration cap, 3 numerical
 *                                   breakdown, 4 unbounded
 *   d_x       n_points x n or NULL  optimal vertex x (NaN unless optimal)
 *   d_dual    n_points x m or NULL  multipliers of the rows: equality rows first (mu), then the inequality rows (lambda >= 0,
 *                                   zero on basic rows), so that c + H theta + A' dual = 0 (NaN unless optimal)
 *   d_active  n_points x words or NULL  final basis: the n - n_eq nonbasic inequality slacks, as a candidate mask
 *   d_iters   n_points x 2 int32 or NULL  pivots of both phases, pivots of Phase 1
 * Asynchronous on `stream`.  Returns -2 for an mpQP handle and for an mpLP whose reduced inequality rows have rank below
 * n - n_eq (no vertex). */
int ppgpu_solve_theta_lp_batch(ppgpu_program* prog, const double* d_theta, int64_t n_points, uint8_t* d_status, double* d_x,
                               double* d_dual, uint64_t* d_active, int32_t* d_iters, ppgpu_stream stream);

/* ---- Mixed-integer programs at fixed theta, by binary assignment y (MixedIntegerThetaSolver of ppopt_b200/mi_theta.py).
 * The handle is the continuous program: the rows that contain a continuous variable, at y = 0.  y enters it the way theta
 * does (right-hand side b + F theta + Fy y with Fy = -A_y; linear term c + H theta + Hy y with Hy the symmetrised Q_xy, zero
 * for an mpMILP).
 *
 * The y columns of the maps the kernels read, reduced with reduce_program's theta-column formulas (host):
 *   h_Fy  m x ny, h_Hy  n x ny or NULL (zero), row major
 *   h_maps  rows x ny, rows = mi + 2 n (mpQP: [V_y | Xp_y | Hy]) or 2 mi + n (mpLP: [Dth_y | Ft_y | X0t_y]); NULL: only
 *           *h_rows is set.
 * Returns -2 when the handle is outside K8 / K9 (see ppgpu_solve_theta_batch / ppgpu_solve_theta_lp_batch). */
int ppgpu_program_param_maps(ppgpu_program* prog, int32_t ny, const double* h_Fy, const double* h_Hy, double* h_maps,
                             int32_t* h_rows);

/* Per assignment a (bit k of d_assign[a] is y_k, nb <= 63): d_off[a][r] = d_base[r] + sum_k d_maps[r][k] y_k (d_base may be
 * NULL), plus 1/2 y' Qyy y on row quad_row when d_qyy (nb x nb) is given.  d_off: n_assign x rows.  Stateless. */
int ppgpu_mi_offsets(const double* d_maps, const double* d_base, int32_t rows, int32_t nb, const uint64_t* d_assign,
                     int64_t n_assign, const double* d_qyy, int32_t quad_row, double* d_off, ppgpu_stream stream);

/* K8 / K9 pair mode: one warp per (point, assignment) pair p = (d_pairs[2p], d_pairs[2p + 1]), the assignment's terms at
 * d_off + d_pairs[2p + 1] * off_ld (the first rows of ppgpu_mi_offsets' output, in the order of ppgpu_program_param_maps).
 * Outputs are per pair and have the meaning of ppgpu_solve_theta_batch / ppgpu_solve_theta_lp_batch's (x the continuous
 * variables of the handle); every one but d_status may be NULL.  d_obj: the continuous part of the objective,
 * 1/2 x'Qx + (c + H theta + Hy y)' x, computed in the warp (NaN unless optimal).  Pass 1 of a batch asks for status and
 * objective only; pass 2 re-solves the winning pair of each point with the full outputs (the same pair gives the same
 * result).  ppgpu_solve_pairs_qp needs an mpQP handle with use_gram, ppgpu_solve_pairs_lp an mpLP handle with a vertex
 * (-2 otherwise). */
int ppgpu_solve_pairs_qp(ppgpu_program* prog, const double* d_theta, const int32_t* d_pairs, int64_t n_pairs, const double* d_off,
                         int64_t off_ld, uint8_t* d_status, double* d_obj, double* d_x, double* d_dual, uint64_t* d_active,
                         int32_t* d_iters, ppgpu_stream stream);
int ppgpu_solve_pairs_lp(ppgpu_program* prog, const double* d_theta, const int32_t* d_pairs, int64_t n_pairs, const double* d_off,
                         int64_t off_ld, uint8_t* d_status, double* d_obj, double* d_x, double* d_dual, uint64_t* d_active,
                         int32_t* d_iters, ppgpu_stream stream);

/* The winner over one chunk of assignments a0 .. a0 + na - 1 (pass-1 outputs d_pair_status / d_pair_obj, n_points x na),
 * folded into a running state per point (d_best = +inf, d_second = +inf, d_best_idx = -1, d_flags = 0 before the first
 * chunk).  A pair counts when its binary-only rows hold at theta (rows of d_off[a] from seg: mb right-hand sides
 * b_i - A_{i,y} y, then H_y' y (t), then the constant c_y'y + 1/2 y'Qyy y; d_Fb mb x t, d_beq mb equality flags) and it is
 * optimal; its objective is d_pair_obj + the constant + theta' H_y' y.  Strict minimum in assignment order (exact ties: the
 * lowest index), d_second the runner-up.  d_status (PPG_MI_* of csrc/tolerances.h) is the status after the chunks so far:
 * unbounded if any counted pair is unbounded, else failed if any hit the iteration cap or broke down, else optimal if any is
 * optimal, else infeasible.  Stateless. */
int ppgpu_mi_select(const double* d_theta, int64_t n_points, int32_t t, const uint8_t* d_pair_status, const double* d_pair_obj,
                    int64_t a0, int32_t na, const double* d_off, int64_t off_ld, int32_t seg, int32_t mb, const double* d_Fb,
                    const uint8_t* d_beq, double* d_best, double* d_second, int32_t* d_best_idx, uint8_t* d_flags,
                    uint8_t* d_status, ppgpu_stream stream);

/* Batched Chebyshev balls of polytopes {theta : E theta <= f} (chebyshev_ball, utils/chebyshev_ball.py:10-63: max r subject to
 * E_i theta + |E_i| r <= f_i): CriticalRegion.is_full_dimension (critical_region.py:89-105, radius > 1e-8) and the Chebyshev /
 * feasibility checks of the program constructor's warnings() (mplp_program.py:162-215).  Stateless - no program handle.
 *   d_rows     total_rows x (t + 1)   stacked rows [f | E] of all polytopes
 *   d_row_off  n_polytopes + 1        first row of every polytope;  max_rows = the largest row count
 *   d_radius   n_polytopes            Chebyshev radius (+inf: unbounded, -inf: empty because of a row 0 <= f < 0)
 *   d_code     n_polytopes int32      PPG_LP_* of csrc/tolerances.h (0 optimal, 2 unbounded, 3 empty, 4 iteration limit) */
int ppgpu_chebyshev_batch(const double* d_rows, const int64_t* d_row_off, int64_t n_polytopes, int32_t t, int32_t max_rows,
                          double* d_radius, int32_t* d_code, ppgpu_stream stream);

/* K10: Chebyshev balls of facets.  For facet p = (d_facets[2p], d_facets[2p+1]) = (polytope, row i of that polytope):
 *   max r  s.t.  a_j theta + |P a_j| r <= f_j  (every other row j of the polytope),  a_i theta = f_i,   P = I - n n', n = a_i / |a_i|
 * solved as the Chebyshev LP of the facet in t - 1 coordinates of its hyperplane (one warp per facet).  A row parallel to the
 * facet is dropped when it holds on the hyperplane and makes the facet empty when it does not.  Stateless.
 *   d_rows, d_row_off, n_poly, t, max_rows   as ppgpu_chebyshev_batch ([f | E], rows need not be normalised), but
 *             1 <= t <= 14 and max_rows <= 256 (a program handle's envelope)
 *   d_center  n_facets x t    a centre of the largest ball inside the facet (NaN unless optimal; for t = 1 the facet's point
 *                             f_i / a_i whenever it is not empty)
 *   d_radius  n_facets        its radius (+inf unbounded, negative / -inf empty)
 *   d_code    n_facets int32  PPG_LP_* of csrc/tolerances.h (0 optimal, 2 unbounded, 3 empty because of a parallel row,
 *                             4 iteration limit), -1 when (polytope, row) is not in the batch.  t = 1: 2 or 3, no LP. */
int ppgpu_facet_chebyshev_batch(const double* d_rows, const int64_t* d_row_off, int64_t n_poly, int32_t t, int32_t max_rows,
                                const int64_t* d_facets, int64_t n_facets, double* d_center, double* d_radius,
                                int32_t* d_code, ppgpu_stream stream);

/* The relaxation tree of a mixed-integer program (mpMILP / mpMIQP): which assignments of the binaries have a feasible
 * relaxation.  Replaces the reference's MITree.__init__ / get_full_leafs (mitree.py) and, at the leaves, its
 * check_bin_feasibility (mpmilp_program.py); the reference runs a MILP per node with Gurobi, here an inner node answers
 * the LP RELAXATION of its partial assignment (sound pruning: an infeasible relaxation has no feasible leaf below it) and a
 * leaf, where every binary is fixed, answers exactly the LP the MILP reduces to.  A handle of its own (csrc/k11_mitree.cu):
 * none of ppgpu_program_create's limits apply.
 *
 * The lifted LP: variables z = (x, theta) (n + t, x in program order), rows A x - F theta <= b (= b on the equality rows
 * 0..n_eq-1 of dims), A_t theta <= b_t, and y_k <= u_k, -y_k <= -l_k for every binary y_k = x[binary_indices[k]].  The
 * root relaxes every binary to [0, 1]; a node at depth d fixes y_k (k < d) to bit k of its uint64.  A node is feasible iff
 * its relaxation has a point within PPG_FEAS_TOL (1 + |rhs|) on every row (csrc/tolerances.h, PPG_TREE_*).
 *   create   dims (n, t, m, q, n_eq; is_qp ignored: the objective plays no part), binary_indices (nb <= 63 column indices of
 *            A), the arrays of ppgpu_program_create.  Returns -2 (ppgpu_last_error says why) when the equalities are rank
 *            deficient, when the lifted rows have rank below the n + t - n_eq free variables (no vertex), or when the
 *            lifted system exceeds the kernel's envelope: (m - n_eq) + q + 2 nb <= 256 rows, n + t - n_eq <= 64 columns.
 *   eval     d_nodes (n uint64) at `depth`: d_status (n uint8: 0 feasible, 1 infeasible, 2 iteration cap, 3 numerical
 *            breakdown), d_point (n x (n + t) or NULL: the feasible point, NaN elsewhere), d_iters (n int32 or NULL:
 *            pivots of the node's LP, -1 when the node inherited its parent's point).  d_parent_point / d_parent_of (or
 *            NULL): the points of the previous depth's eval and, per node, the index of its parent there
 *            (ppgpu_tree_children writes it); when given and inheritance is on, a node whose parent's point, with y_{depth-1}
 *            snapped to the node's value, satisfies every row is feasible without an LP.  Statuses do not depend on it.
 *   children the nodes with status 0 in order (d_idx, n int64 scratch), each followed by its two children at depth + 1:
 *            d_children[2j] fixes y_depth = 0, d_children[2j + 1] fixes it to 1 (2n uint64), d_parent_of the index of the
 *            parent (2n int64); h_count = number of feasible parents.  d_ws: ppgpu_select_workspace_bytes(n) bytes.
 *            Synchronises the stream. */
typedef struct ppgpu_tree ppgpu_tree;
int ppgpu_tree_create(const ppgpu_dims* dims, const int32_t* h_binary_indices, int32_t nb, const double* h_A, const double* h_b,
                      const double* h_F, const double* h_A_t, const double* h_b_t, int device, ppgpu_tree** out);
int ppgpu_tree_destroy(ppgpu_tree* tree);
/*   PPGPU_TREE_OPT_INHERIT  1 / 0 (default; the environment's PPGPU_TREE_INHERIT at create): point inheritance on / off */
#define PPGPU_TREE_OPT_INHERIT 0
int ppgpu_tree_set_option(ppgpu_tree* tree, int32_t option, int64_t value);
int ppgpu_tree_eval(ppgpu_tree* tree, const uint64_t* d_nodes, int64_t n, int32_t depth, uint8_t* d_status, double* d_point,
                    const double* d_parent_point, const int64_t* d_parent_of, int32_t* d_iters, ppgpu_stream stream);
int ppgpu_tree_children(ppgpu_tree* tree, const uint64_t* d_nodes, const uint8_t* d_status, int64_t n, int32_t depth,
                        int64_t* d_idx, uint64_t* d_children, int64_t* d_parent_of, int64_t* h_count, void* d_ws,
                        size_t ws_bytes, ppgpu_stream stream);

/* cumulative device counters (LPs, pivots, useful FMAs per kernel family, borderline/numeric flags) */
int ppgpu_counters(ppgpu_program* prog, uint64_t* h_out, int32_t reset, ppgpu_stream stream);

/* how many kernels this library has launched on behalf of the handle since creation */
int64_t ppgpu_launch_count(const ppgpu_program* prog);

/* Optional per-kernel-family timing with CUDA events recorded on the launch stream (used by bench.py for the
 * roofline line).  Families: 0 K1 rank, 1 K2 feasibility LP, 2 K3/K4 screen, 3 K5 emission, 4 K6 count, 5 K6 write,
 * 6 ordered compaction, 7 K2a relaxation certificates, 8 K2w vertex-walk certificates, 9 certificates inherited from the
 * parents' witnesses.  h_ms / h_launches hold PPGPU_NUM_FAMILIES entries. */
#define PPGPU_NUM_FAMILIES 10
int ppgpu_profile_enable(ppgpu_program* prog, int32_t on);
int ppgpu_profile_read(ppgpu_program* prog, double* h_ms, int64_t* h_launches, int32_t reset);

/* register-resident DFMA loop over all SMs: the FP64 roofline denominator, in TFLOP/s */
int ppgpu_measure_fp64_peak(int32_t iters, double* h_tflops, ppgpu_stream stream);

#ifdef __cplusplus
}
#endif
#endif /* PPGPU_H */
