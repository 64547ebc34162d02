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
cudaError_t launch_k2w(const DevProgram& P, const uint64_t* masks, long long n, int k_act, uint8_t* status,
                       unsigned long long* queue, unsigned long long* counters, int sm_count, cudaStream_t st, bool* handled,
                       uint64_t* witness, int* order_scratch, bool reference);
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
// K8: one fixed-theta QP per point (dual active set on the Gram data, csrc/k8_theta_qp.cu); x / dual / mask / iters may be null
cudaError_t launch_theta_qp(const DevProgram& P, const double* theta, long long n_points, uint8_t* status, double* x,
                            double* dual, uint64_t* mask, int* iters, int sm_count, cudaStream_t st);
// K9: one fixed-theta LP per point (dictionary simplex from the handle's start dictionary, csrc/k9_theta_lp.cu);
// iters (n x 2: pivots, Phase 1 pivots), x / dual / mask / iters may be null
cudaError_t launch_theta_lp(const DevProgram& P, const double* theta, long long n_points, uint8_t* status, double* x,
                            double* dual, uint64_t* mask, int* iters, int sm_count, cudaStream_t st);
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
