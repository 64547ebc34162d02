// Host-side launch entry points of the individual kernels (internal to libppgpu).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "common.cuh"

namespace ppgpu {

// Opt a kernel in to the device's full dynamic shared memory.  Always the SAME value: cudaFuncSetAttribute is per function
// and process wide, and handles are driven from several host threads at once (mpMIQP sub-problems on their own streams) -
// setting the size of the launch at hand let one thread shrink the limit under another thread's launch.
template <class K>
inline cudaError_t allow_max_smem(K kern) {
    int dev = 0, lim = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&lim, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
    if (e != cudaSuccess) return e;
    cudaFuncAttributes fa;
    if ((e = cudaFuncGetAttributes(&fa, kern)) != cudaSuccess) return e;
    return cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, lim - (int)fa.sharedSizeBytes);   // static + dynamic <= limit
}

// Opts in (allow_max_smem) when a launch with `dyn` bytes of dynamic shared memory would exceed the 48 KB a block gets without
// it.  The kernel's static shared memory counts against the same 48 KB: a dynamic size just below 48 KB alone fails with
// "invalid argument" on the first launch of a kernel that also has static arrays.
template <class K>
inline cudaError_t fit_smem(K kern, size_t dyn) {
    cudaFuncAttributes fa;
    const cudaError_t e = cudaFuncGetAttributes(&fa, kern);
    if (e != cudaSuccess) return e;
    return fa.sharedSizeBytes + dyn > 48 * 1024 ? allow_max_smem(kern) : cudaSuccess;
}

// Launch shape of a kernel that runs one warp per item over n items with a grid-stride loop: as many warps per CTA as the
// device's opt-in shared memory holds next to the kernel's static shared memory and `fixed_bytes` of dynamic shared memory
// ahead of the warps' blocks (at most max_warps), the dynamic shared memory that takes, and a grid capped at the CTAs that
// are resident at once.  Opts the kernel in (fit_smem) when the size needs it; cudaErrorInvalidValue when no warp fits.
struct WarpGrid {
    int warps;
    size_t smem;
    unsigned grid;
};
template <class K>
inline cudaError_t warp_grid(K kern, size_t warp_bytes, size_t fixed_bytes, int max_warps, long long n, int sm_count,
                             WarpGrid* out) {
    int dev = 0, lim = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&lim, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
    if (e != cudaSuccess) return e;
    cudaFuncAttributes fa;
    if ((e = cudaFuncGetAttributes(&fa, kern)) != cudaSuccess) return e;
    const size_t used = fa.sharedSizeBytes + fixed_bytes;
    int wpb = used < (size_t)lim ? (int)(((size_t)lim - used) / warp_bytes) : 0;
    if (wpb > max_warps) wpb = max_warps;
    if (wpb < 1) return cudaErrorInvalidValue;
    const size_t smem = fixed_bytes + (size_t)wpb * warp_bytes;
    if ((e = fit_smem(kern, smem)) != cudaSuccess) return e;
    int per_sm = 0;
    if ((e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, wpb * 32, smem)) != cudaSuccess) return e;
    if (per_sm < 1) per_sm = 1;
    long long grid = (n + wpb - 1) / wpb;
    const long long cap = (long long)sm_count * per_sm;
    if (grid > cap) grid = cap;
    *out = {wpb, smem, (unsigned)grid};
    return cudaSuccess;
}

int k2_pad_columns(int ncols_with_rhs);

cudaError_t launch_k1(const DevProgram& P, const uint64_t* masks, long long n, int k_act, uint8_t* status,
                      unsigned long long* counters, int sm_count, cudaStream_t st);
cudaError_t launch_k2(const DevProgram& P, const uint64_t* masks, long long n, uint8_t* status,
                      unsigned long long* queue, unsigned long long* counters, int sm_count, cudaStream_t st);
cudaError_t launch_k2a(const DevProgram& P, const uint64_t* masks, long long n, int k_act, uint8_t* status,
                       unsigned long long* queue, unsigned long long* counters, int max_iter, int sm_count, cudaStream_t st);
cudaError_t launch_k2a_prefix(const DevProgram& P, const uint64_t* masks, long long n, int k_act, uint8_t* status,
                              unsigned long long* queue, unsigned long long* counters, int max_iter, int sm_count,
                              cudaStream_t st, bool* handled);
// K2w: feasibility certificates shared between the candidates of a prefix by a primal-simplex walk over vertices
// witness (n x W, may be null): receives the active-row mask of the vertex that certified a candidate
// prove_infeasible: candidates whose last drive ends at an optimum that proves them infeasible get PPG_ST_PRE (and no
// PPG_ST_FEAS); the caller clears that mark after K2
cudaError_t launch_k2w(const DevProgram& P, const uint64_t* masks, long long n, int k_act, uint8_t* status,
                       unsigned long long* queue, unsigned long long* counters, int sm_count, cudaStream_t st, bool* handled,
                       uint64_t* witness, int* order_scratch, bool reference, bool prove_infeasible);
// ints of scratch launch_k2w wants for ordering the work items of an n-candidate launch (may be passed as null: natural order)
size_t k2w_order_scratch_ints(long long n);
// certificates INHERITED from the previous level: a candidate is feasible when the witness vertex of one of its parents
// (candidate minus one row, looked up in the prefix-group index K6 built for that level) has the dropped row active as well
cudaError_t launch_inherit(const DevProgram& P, const uint64_t* masks, long long n, uint8_t* status, uint64_t* witness_out,
                           const uint64_t* parent_feas, long long parent_nf, const void* parent_ws, const uint64_t* parent_wit,
                           unsigned long long* counters, cudaStream_t st);
cudaError_t launch_k34(const DevProgram& P, const uint64_t* masks, long long n, int k_act, uint8_t* status,
                       unsigned long long* queue, unsigned long long* counters, int sm_count, cudaStream_t st);
cudaError_t launch_k34_compact(const DevProgram& P, const uint64_t* masks, long long n, int k_act, uint8_t* status,
                               unsigned long long* queue, unsigned long long* counters, int sm_count, cudaStream_t st,
                               int use_pre, bool* handled);
// general (LU) path: marks every feasible candidate that the reference would hand to check_optimality
cudaError_t launch_mark_general(const DevProgram& P, long long n, int k_act, uint8_t* status, cudaStream_t st);

// region emission: K5a (KKT, rows, full-dimension test), K5b (redundancy LPs, one warp per LP), K5c (duplicates);
// k5_launches(t) kernels per call
cudaError_t launch_k5(const DevProgram& P, const uint64_t* masks, const long long* idx, long long n_sel, int k_act,
                      double* laws, double* rows, int32_t* flags, double* info, uint8_t* status,
                      unsigned long long* queue, unsigned long long* counters, int sm_count, cudaStream_t st);
int k5_launches(int t);

size_t scan_workspace_bytes(long long n);
size_t select_workspace_bytes(long long n);
const long long* children_order_flag(const void* ws, long long nf);
cudaError_t select_indices(const uint8_t* status, long long n, uint8_t bits, uint8_t value, long long* idx_out,
                           long long* d_count, void* ws, size_t ws_bytes, cudaStream_t st);
cudaError_t root_level(const DevProgram& P, uint64_t* masks, long long* d_count, cudaStream_t st);
cudaError_t children_count(const DevProgram& P, const uint64_t* masks, const long long* feas_idx, long long nf,
                           int k_act, uint64_t* feas_masks, uint64_t* survive, long long* offsets, void* ws,
                           size_t ws_bytes, unsigned long long* counters, cudaStream_t st);
cudaError_t children_prepare(const DevProgram& P, const uint64_t* masks, const long long* feas_idx, long long nf,
                             uint64_t* feas_masks, void* ws, size_t ws_bytes, cudaStream_t st);
cudaError_t children_count_range(const DevProgram& P, const uint64_t* feas_masks, long long nf, int k_act, uint64_t* survive,
                                 long long* counts, long long p_lo, long long p_hi, void* ws, unsigned long long* counters,
                                 cudaStream_t st);
cudaError_t children_scan(long long* counts_to_offsets, long long nf, void* ws, cudaStream_t st);
cudaError_t children_write(const DevProgram& P, const uint64_t* feas_masks, const uint64_t* survive,
                           const long long* offsets, long long nf, uint64_t* children, cudaStream_t st);

cudaError_t launch_locate(const double* theta, long long n_points, int t, const double* rows, const long long* row_off,
                          long long n_regions, const double* laws, int n_x, int use_tol, double tol, int overlap,
                          const double* Qm, const double* Hm, const double* cv, int* region_out, double* x_out, int sm_count,
                          cudaStream_t st);

cudaError_t launch_cheb_batch(const double* rows, const long long* row_off, long long n_poly, int t, int max_rows,
                              double* radius, int* code, int sm_count, cudaStream_t st);
// K10: Chebyshev balls of facets (polytope, row) of stacked polytopes (csrc/k34c_compact.cu)
cudaError_t launch_facet_cheb(const double* rows, const long long* row_off, long long n_poly, int t, int max_rows,
                              const long long* facets, long long n_facets, double* center, double* radius, int* code,
                              int sm_count, cudaStream_t st);
// K8: one fixed-theta QP per point (dual active set on the Gram data, csrc/k8_theta_qp.cu); x / dual / mask / iters may be null
cudaError_t launch_theta_qp(const DevProgram& P, const double* theta, long long n_points, uint8_t* status, double* x,
                            double* dual, uint64_t* mask, int* iters, int sm_count, cudaStream_t st);
// K9: one fixed-theta LP per point (dictionary simplex from the handle's start dictionary, csrc/k9_theta_lp.cu);
// iters (n x 2: pivots, Phase 1 pivots), x / dual / mask / iters may be null
cudaError_t launch_theta_lp(const DevProgram& P, const double* theta, long long n_points, uint8_t* status, double* x,
                            double* dual, uint64_t* mask, int* iters, int sm_count, cudaStream_t st);
// K8 / K9 pair mode (PairArgs of common.cuh): one warp per (point, assignment) pair, outputs per pair; all but status may be null
cudaError_t launch_theta_qp_pairs(const DevProgram& P, const double* theta, const PairArgs& pa, long long n_pairs, uint8_t* status,
                                  double* x, double* dual, uint64_t* mask, int* iters, int sm_count, cudaStream_t st);
cudaError_t launch_theta_lp_pairs(const DevProgram& P, const double* theta, const PairArgs& pa, long long n_pairs, uint8_t* status,
                                  double* x, double* dual, uint64_t* mask, int* iters, int sm_count, cudaStream_t st);
// per assignment a (bit k of assign[a] = y_k): off[a][r] = base[r] + sum_k maps[r][k] y_k, plus 1/2 y'Qyy y on row quad_row
cudaError_t launch_mi_offsets(const double* maps, const double* base, int rows, int nb, const uint64_t* assign, long long n_assign,
                              const double* qyy, int quad_row, double* off, cudaStream_t st);
// the running minimum over assignments a0 .. a0 + na - 1 per point (csrc/mi_theta.cu)
struct MiSelectArgs {
    const double* theta; long long n_points; int t;
    const uint8_t* pair_status; const double* pair_obj;   // n_points x na
    long long a0; int na;
    const double* off; long long off_ld; int seg;         // off[a][seg ..]: binary-row rhs (mb), H_y' y (t), constant (1)
    int mb; const double* Fb; const uint8_t* beq;          // binary-only rows: F (mb x t), equality flags
    double* best; double* second; int* best_idx; uint8_t* flags; uint8_t* status;
};
cudaError_t launch_mi_select(const MiSelectArgs& a, cudaStream_t st);
// K11: the relaxation tree of a mixed-integer program (csrc/k11_mitree.cu, lifted system of host_math.hpp::TreeProgram).
// Nodes are uint64 with bit k = y_k for k < depth.
struct DevTree {
    int nv, rows, cols, rb0, tp, ld, ne, nb;
    const double* D0;      // rows x ld  [beta0 | D | Dbnd]
    const int* bvar;       // rows
    const int* nvar;       // cols
    const double* hs;      // rows
    const double* z0;      // nv
    const double* Q2;      // nv x cols
    const double* Arows;   // (ne + rows) x nv
    const double* brows;   // ne + rows
    const int* bin;        // nb
};
// status (PPG_TREE_*), point (n x nv, NaN unless feasible) and iters (pivots) may be null except status; skip_done: nodes
// whose status is already PPG_TREE_FEASIBLE (certified by inheritance) are left as they are
cudaError_t launch_tree_node(const DevTree& P, const uint64_t* nodes, long long n, int depth, uint8_t* status, double* point,
                             int* iters, int skip_done, int sm_count, cudaStream_t st);
// one thread per node at `depth` >= 1: the parent's point with y_{depth-1} snapped to the node's value; certified ->
// status PPG_TREE_FEASIBLE, the snapped point and iters = -1; otherwise status PPG_TREE_UNDECIDED
cudaError_t launch_tree_inherit(const DevTree& P, const uint64_t* nodes, long long n, int depth, const double* parent_point,
                                const long long* parent_of, uint8_t* status, double* point, int* iters, cudaStream_t st);
// children of the selected nodes idx[0..*d_count) (n_max bounds the count): 2j fixes y_depth = 0, 2j + 1 fixes it to 1
cudaError_t launch_tree_children(const uint64_t* nodes, const long long* idx, const long long* d_count, long long n_max, int depth,
                                 uint64_t* children, long long* parent_of, cudaStream_t st);
cudaError_t launch_clear_bits(uint8_t* status, long long n, uint8_t bits, cudaStream_t st);

cudaError_t measure_fp64_peak(int iters, double* tflops, cudaStream_t st);

}  // namespace ppgpu
