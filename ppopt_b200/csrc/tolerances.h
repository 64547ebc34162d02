// Decision thresholds of the combinatorial path. Shared by the CUDA kernels and the CPU checker.
//
// Literal reference constants (must not be tuned):
//   PPG_ZERO_ROW   all |a_ij| <= 1e-8  -> numerically zero row   (utils/constraint_utilities.py:469-470)
//   PPG_RADIUS     Chebyshev radius > 1e-8 -> full dimensional    (utils/mpqp_utils.py:343)
//   PPG_WIDTH_1D   min + 1e-8 <= max                              (utils/mpqp_utils.py:320)
// LP-backend behaviour that the reference inherits from GLPK/HiGHS (primal feasibility tolerance):
//   PPG_FEAS_TOL   a row may be violated by at most 1e-7
// Engine-internal numerics (pivoting / anti-cycling), no reference counterpart:
//   PPG_PIV_TOL, PPG_OPT_TOL, PPG_HARRIS, PPG_DEGEN_STEP, PPG_BLAND_AFTER, PPG_RANK_TOL
#pragma once

#define PPG_ZERO_ROW 1e-8
#define PPG_RADIUS 1e-8
#define PPG_WIDTH_1D 1e-8
#define PPG_FEAS_TOL 1e-7
// redundancy LPs of gen_cr_from_active_set (mpqp_utils.py:143-178): a row is kept iff its hyperplane touches the
// region.  Calibrated on the runnable reference (HiGHS with presolve): it drops rows whose best margin is
// <= -2.7e-8 and keeps rows down to -4.8e-14 on every fixture except the stacked control-allocation family,
// where its own decisions overlap in [-2.3e-8, 5e-11] (DESIGN.md "weakly redundant rows").
#define PPG_REDUND_TOL 1e-9
// the Gram/Cholesky screen (K3/K4) passes candidates with half the radius to the LU-based final test
#define PPG_RADIUS_SCREEN 0.5e-8
// The reference decides "full dimensional" by comparing a radius that ITS LP BACKEND computed with 1e-8
// (mpqp_utils.py:343), and that backend only guarantees its answer to its own feasibility tolerance (1e-7): on
// ctrl_alloc_n5 level 4 HiGHS reports 2.78e-8 for 26 polytopes whose exact radius is -7.78e-9 (50-digit
// arithmetic, DESIGN.md section 5).  The engine decides with the accurate radius and raises PPG_ST_THIN on every
// candidate whose radius lies within this band of the threshold, so that the discrepancy is never silent.
#define PPG_RADIUS_BAND 1e-7

// Infeasibility certificate of the vertex walk (csrc/k2w_walk.cu).  A drive of row b that stops with every free
// coefficient of its row <= 0 proves that the feasibility LP of its candidate (K2: max s with every slack >= s and the
// candidate's slacks = 0) has s* <= -beta_b / sum_free |D_bj|.  The walk decides "infeasible" only when
//     beta_b - PPG_WALK_INF_REL * (1 + |beta_b|) > PPG_WALK_INF_MARGIN * sum_free |D_bj|
// i.e. when that bound clears K2's threshold (-PPG_FEAS_TOL) ten times over, after an allowance for the rounding of the
// walk's beta.  Measured drift of the walk's dictionary before it is reloaded (DESIGN.md section 3): 9e-14 absolute on D,
// 1e-13 relative on beta after 2,400 pivots.  The allowance is relative to |beta_b| because the programs carry box rows of
// 1e7 next to rows near 1 (an absolute error of 1e-6 on such a row is still 1e-13 relative); 1e-9 keeps four orders of
// magnitude over the measured drift.  The factor ten on PPG_FEAS_TOL covers K2's own rounding.  Bounds inside the band are
// left to K2a and K2.
#define PPG_WALK_INF_MARGIN (10 * PPG_FEAS_TOL)
#define PPG_WALK_INF_REL 1e-9

#define PPG_PIV_TOL 1e-9
#define PPG_OPT_TOL 1e-12  // reduced-cost threshold: the objective error is tol x distance travelled (theta ranges of 1e2), so 1e-9 was too loose
#define PPG_HARRIS 1e-9
#define PPG_TINY 1e-12   // entries below this are treated as structural zeros in the ratio test
#define PPG_DEGEN_STEP 1e-12
#define PPG_BLAND_AFTER 8
// column-pivoted QR: rank deficient iff |R_kk| <= PPG_RANK_TOL * |R_11|
// (numpy.linalg.matrix_rank default: sigma_min <= sigma_max * max(k,n) * eps, constraint_utilities.py:236)
#define PPG_RANK_TOL 1e-11
#define PPG_RANK_BORDER_LO 1e-15   // below: exactly dependent rows (3e-16 on the MPC programs); above: re-decided by singular values
#define PPG_RANK_BORDER_HI 1e-7

// per-candidate status byte (bits 0-3 match tests/golden level*_status)
#define PPG_ST_RANK 1u      // LICQ holds: rank(A_active) == |active|
#define PPG_ST_FEAS 2u      // feasibility LP has a solution
#define PPG_ST_OPT 4u       // passed the optimality screen (theta-space polytope non-empty, full-dimensional)
#define PPG_ST_REGION 8u    // a critical region was emitted
#define PPG_ST_BORDER 16u   // a decision fell inside a borderline band (reported, never silently ignored)
#define PPG_ST_NUMERIC 32u  // iteration limit / singular KKT / non-finite value
#define PPG_ST_THIN 64u     // full-dimension decision taken inside PPG_RADIUS_BAND of the 1e-8 threshold (reported)
#define PPG_ST_PRE 128u       // transient: passed the K3 thread-per-candidate prefilter (cleared by k34_kernel); before
                              // that, in the feasibility stage: handed over by K2a, or proved infeasible by the vertex walk
                              // (cleared after K2)

// witness slots per candidate (ppgpu_level_eval_w): [0] the vertex that certified it (walk or inheritance), [1..] later
// vertices of the walk that hold it as well, written in turn.  Measured on the bench program (share of level 5 that inherits /
// ms per step): 1 slot 73 % / 240.7, 2 slots 85.5 % / 223.9, 3 slots 87.3 % / 220.3 - two it is (16 B per slot and candidate).  Also measured and rejected: slot 1 as the UNION of all
// later vertices (a "cover": certifies as well, but names no vertex a child could pass on - 82 % / 239.8; as a third slot
// next to two vertices 85.6 % / 230.5)
#define PPG_WITNESS_SLOTS 2

// LP return codes
#define PPG_LP_OPTIMAL 0
#define PPG_LP_EARLY 1
#define PPG_LP_UNBOUNDED 2
#define PPG_LP_INFEAS_EQ 3
#define PPG_LP_ITERLIM 4

// K8 fixed-theta QP (dual active set on  w = G lambda + V [1; theta],  csrc/k8_theta_qp.cu), shared with the CPU twin.
// Engine-internal numerics, no reference counterpart (the reference hands the QP to daqp / gurobi / ...):
//   PPG_QP_TOL       row j is violated when w_j < -PPG_QP_TOL * (1 + |V_j [1; theta]|) (its own scale: programs carry
//                    big-M rows of 1e7 next to rows of 1e-3); optimal when no row outside W is violated
//   PPG_QP_CURV      a constraint is added only when its curvature z = G_jj - |L^-1 G_Wj|^2 exceeds PPG_QP_CURV * G_jj
//   PPG_QP_DTOL      a working-set multiplier blocks the step only when it falls at rate d_i < -PPG_QP_DTOL
//   PPG_QP_MAX_ITER  steps (adds + drops) per point before the point is reported with status PPG_QP_ITERLIM
#define PPG_QP_TOL 1e-10
#define PPG_QP_CURV 1e-10
#define PPG_QP_DTOL 1e-12
#define PPG_QP_MAX_ITER 1000
// status per point
#define PPG_QP_OPTIMAL 0
#define PPG_QP_INFEASIBLE 1
#define PPG_QP_ITERLIM 2
#define PPG_QP_NUMERIC 3

// K9 fixed-theta LP (dense primal dictionary simplex from the theta-independent start of host_math.hpp::build_lp_dictionary,
// csrc/k9_theta_lp.cu).  Engine-internal numerics, no reference counterpart (the reference hands the LP to GLPK / HiGHS / ...):
//   PPG_TLP_TOL       feasibility tolerance of slack i: delta_i = PPG_TLP_TOL * (1 + |bti_i + Ft_i theta|), the scale of the
//                     row's own right-hand side (as K8's PPG_QP_TOL): the synthetic programs carry box rows of 1e7 next to
//                     rows near 1, and one absolute tolerance is either meaningless on the first or too loose on the second
//                     (the start dictionary's beta is no scale: the start vertex can lie far outside the feasible set).
//                     delta_i is the Harris relaxation of the row in the ratio test and the margin below which Phase 1
//                     starts at all; x0 > delta of the slack x0 entered on ends Phase 1 as infeasible
//   PPG_TLP_OPT       reduced-cost threshold: Phase 2 is optimal when every d_j <= PPG_TLP_OPT * (1 + max_i |c_i + H_i theta|)
//                     (the cost vector's own scale); Phase 1 uses it unscaled (the auxiliary row starts with coefficients -1)
//   PPG_TLP_TINY      column entries at or below this do not block the ratio test (structural zeros left by elimination)
//   PPG_TLP_PIV       a basic auxiliary variable at zero is pivoted out on its largest entry only when that exceeds this
//   PPG_TLP_MAX_ITER  pivots per point (both phases) before the point is reported with PPG_TLP_ITERLIM; Bland's rule
//                     (after PPG_BLAND_AFTER degenerate pivots) excludes cycling, so the cap is a guard against numerical
//                     stalling only: a vertex path of a 256-row dictionary is far shorter
#define PPG_TLP_TOL 1e-10
#define PPG_TLP_OPT 1e-12
#define PPG_TLP_TINY 1e-12
#define PPG_TLP_PIV 1e-9
#define PPG_TLP_MAX_ITER 4000
// status per point: 0-3 mean what PPG_QP_* means
#define PPG_TLP_OPTIMAL 0
#define PPG_TLP_INFEASIBLE 1
#define PPG_TLP_ITERLIM 2
#define PPG_TLP_NUMERIC 3
#define PPG_TLP_UNBOUNDED 4

// K11 relaxation tree of an mpMIQP / mpMILP (Phase 1 of the lifted LP per node, csrc/k11_mitree.cu).  A node is feasible iff
// its relaxation has a point z with  a_i z - h_i <= PPG_FEAS_TOL (1 + |h_i|)  on every row (|.| on the equality rows), h_i the
// row's right-hand side at the node's bounds.  Phase 1 splits that budget: the Harris relaxation of a slack row is half of it
// and x0 (Chvatal's auxiliary column) must end at or below PPG_TREE_AUX = half of PPG_FEAS_TOL, so the point read off a
// feasible node's final dictionary violates row i by at most PPG_FEAS_TOL (1 + |h_i|).  An inherited point is certified
// against the full PPG_FEAS_TOL (1 + |h_i|) of every row.  Pivoting rules and the other thresholds are K9's (PPG_TLP_*).
#define PPG_TREE_HARRIS 0.5e-7
#define PPG_TREE_AUX 0.5e-7
// status per node: 0-3 mean what PPG_TLP_* means (feasible / infeasible / iteration cap / numerical breakdown)
#define PPG_TREE_FEASIBLE 0
#define PPG_TREE_INFEASIBLE 1
#define PPG_TREE_UNDECIDED 255   // transient: the inheritance check did not certify the node, the LP decides it

// ---- fixed-theta solves of a mixed-integer program by assignment (K8 / K9 pair mode, csrc/mi_theta.cu)
//   PPG_MI_ROW_TOL   a binary-only row (no continuous variable) holds at (theta, y) when b_i + F_i theta - A_{i,y} y >=
//                    -PPG_MI_ROW_TOL * (1 + |.|) (an equality row: |.| <= that), the tolerance of the relaxation tree
#define PPG_MI_ROW_TOL 1e-7
// status per point: the winner is optimal; no pair is feasible; some pair hit the iteration cap or broke down (the minimum
// is not certified); some feasible pair is unbounded (mpMILP)
#define PPG_MI_OPTIMAL 0
#define PPG_MI_INFEASIBLE 1
#define PPG_MI_FAILED 2
#define PPG_MI_UNBOUNDED 4
// running flags of mi_select
#define PPG_MI_ANY_OPTIMAL 1
#define PPG_MI_ANY_FAILED 2
#define PPG_MI_ANY_UNBOUNDED 4
