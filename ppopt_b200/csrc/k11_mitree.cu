// K11 - the relaxation tree of a mixed-integer program (mpmiqp_enumeration's screen of the binary assignments).
//
// A node at depth d fixes y_0..y_{d-1}; it is feasible iff the LP relaxation of the lifted system (host_math.hpp::TreeProgram:
// z = (x, theta), the program's rows, Theta's rows and two bound rows per binary) has a point within PPG_FEAS_TOL.  The
// dictionary entries are the same for every node; only the right-hand side depends on the node's bounds.
//
// k11_tree_node_kernel, one warp per node, grid-stride:
//   1. copies the dictionary into the warp's shared memory with the auxiliary column x0 of warp_dict.cuh, evaluates
//      beta(node) = beta0 + sum_{k<d} Dbnd[:, 2k + y_k] and the Harris relaxation of every slack, PPG_TREE_HARRIS (1 + |h_i|)
//      with h_i the row's right-hand side at the node;
//   2. Phase 1 only, with the rules of warp_dict.cuh: when some slack row is below its relaxation, x0 enters, then the x0 row
//      is minimised.  Feasible as soon as x0 leaves or when the minimum is at most PPG_TREE_AUX (x0's tolerance);
//      infeasible when it is larger.
//   Outputs: a status byte, the pivot count and, when asked for, the point z = z0 + Q2 v of the final dictionary.
// k11_tree_inherit_kernel, one thread per node: the parent's point with the newly fixed binary snapped to the node's value is
//   checked against every lifted row at the node's bounds with the verdict's tolerance; when it holds, the node is feasible
//   without an LP and inherits that point.  It never decides infeasibility.
// k11_tree_children_kernel, one thread per selected (feasible) node: children in parent order, y_d = 0 before y_d = 1, so
//   the leaves come out in lexicographic order of (y_0, y_1, ...).
#include <cmath>

#include "common.cuh"
#include "launch.h"
#include "warp_dict.cuh"

namespace ppgpu {

constexpr int K11_MAX_WARPS = 16;

__host__ __device__ inline WarpDictLayout k11_layout(int rows, int cols) { return warp_dict_layout(rows, rows, cols, 0); }

// scale 1 + |h_i| of inequality row s at a node: the bound rows of the fixed binaries have h = y_k (upper) and -y_k (lower)
__device__ __forceinline__ double k11_scale(const DevTree& P, int s, uint64_t node, int depth) {
    const int k = (s - P.rb0) >> 1;
    if (s >= P.rb0 && k < depth) return 1.0 + (double)((node >> k) & 1ull);
    return __ldg(P.hs + s);
}

__global__ void __launch_bounds__(K11_MAX_WARPS * 32)
k11_tree_node_kernel(DevTree P, const uint64_t* __restrict__ nodes, long long n, int depth, uint8_t* __restrict__ status_out,
                     double* __restrict__ point_out, int* __restrict__ iters_out, int skip_done) {
    extern __shared__ double k11_smem[];
    const int rows = P.rows, cols = P.cols, ld0 = P.ld, nv = P.nv;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, wpb = blockDim.x >> 5;
    const WarpDictLayout lo = k11_layout(rows, cols);
    const int LD = lo.LD, nc = cols + 1, AUX = rows;   // nonbasic columns 0..cols (column cols starts as x0); x0's id
    double* base = k11_smem + (size_t)warp * lo.stride;
    double* T = base + lo.T;
    double* Pr = base + lo.P;
    double* tolv = base + lo.tol;
    int* bvar = (int*)(base + lo.bvar);
    int* nvar = (int*)(base + lo.nvar);
    const double QNAN = __longlong_as_double(0x7ff8000000000000ll);

    for (long long pt = (long long)blockIdx.x * wpb + warp; pt < n; pt += (long long)gridDim.x * wpb) {
        if (skip_done && status_out[pt] == PPG_TREE_FEASIBLE) continue;   // warp-uniform: every lane reads the same byte
        const uint64_t node = nodes[pt];
        __syncwarp();
        // constant entries: row by row, lanes over the columns (coalesced reads of the start dictionary)
        for (int r = 0; r < rows; ++r)
            for (int c = lane; c < cols; c += 32) T[(size_t)r * LD + 1 + c] = __ldg(P.D0 + (size_t)r * ld0 + 1 + c);
        for (int r = lane; r < rows; r += 32) {
            const double* src = P.D0 + (size_t)r * ld0;
            double b = __ldg(src);
            for (int k = 0; k < depth; ++k) b += __ldg(src + 1 + cols + 2 * k + (int)((node >> k) & 1ull));
            const int bv = __ldg(P.bvar + r);
            T[(size_t)r * LD] = b;
            T[(size_t)r * LD + 1 + cols] = bv >= 0 ? -1.0 : 0.0;
            bvar[r] = bv;
            tolv[r] = PPG_TREE_HARRIS * k11_scale(P, r, node, depth);   // by slack id (slack r starts in row r)
        }
        for (int c = lane; c < cols; c += 32) nvar[c] = __ldg(P.nvar + c);
        if (lane == 0) nvar[cols] = AUX;
        __syncwarp();

        WarpDict wd{T, Pr, tolv, bvar, nvar, LD, rows, rows, nc, lane, PPG_TREE_AUX};
        int status = -1;
        const int aux_row = wd.x0_row();
        if (aux_row == WD_NONE) status = PPG_TREE_FEASIBLE;
        else if (!wd.pivot(aux_row, cols)) status = PPG_TLP_NUMERIC;
        while (status < 0) {
            const double* orow = T + (size_t)aux_row * LD;
            const int j = wd.price(orow, PPG_TLP_OPT);
            if (j == WD_NONE) { status = orow[0] > wd.aux_tol ? PPG_TREE_INFEASIBLE : PPG_TREE_FEASIBLE; break; }
            if (wd.it >= PPG_TLP_MAX_ITER) { status = PPG_TLP_ITERLIM; break; }
            const WarpDict::Ratio q = wd.ratio(j, aux_row);
            // x0's row blocks every column that decreases it: a test that blocks nothing is a breakdown
            if (!q.blocked || q.row == WD_NONE) { status = PPG_TLP_NUMERIC; break; }
            wd.count_step(q.step);
            if (!wd.pivot(q.row, j)) { status = PPG_TLP_NUMERIC; break; }
            if (q.row == aux_row) { status = PPG_TREE_FEASIBLE; break; }
        }
        status = wd.settle(status, PPG_TREE_FEASIBLE);
        if (lane == 0) status_out[pt] = (uint8_t)status;
        if (iters_out && lane == 0) iters_out[pt] = wd.it;
        if (!point_out) continue;
        if (status != PPG_TREE_FEASIBLE) {
            for (int i = lane; i < nv; i += 32) point_out[pt * nv + i] = QNAN;
            continue;
        }
        // v from its rows (staged in the pivot row), z = z0 + Q2 v
        wd.stage_v();
        for (int i = lane; i < nv; i += 32) {
            double v = __ldg(P.z0 + i);
            for (int c = 0; c < cols; ++c) v = fma(__ldg(P.Q2 + (size_t)i * cols + c), Pr[c], v);
            point_out[pt * nv + i] = v;
        }
    }
}

__global__ void k11_tree_inherit_kernel(DevTree P, const uint64_t* __restrict__ nodes, long long n, int depth,
                                        const double* __restrict__ parent_point, const long long* __restrict__ parent_of,
                                        uint8_t* __restrict__ status_out, double* __restrict__ point_out, int* __restrict__ iters_out) {
    const long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    const int nv = P.nv, ne = P.ne, k = depth - 1;
    const uint64_t node = nodes[j];
    const double* z = parent_point + (size_t)parent_of[j] * nv;
    const int col = __ldg(P.bin + k);
    const double yk = (double)((node >> k) & 1ull);
    bool ok = !isnan(z[0]);
    for (int i = 0; ok && i < ne + P.rows; ++i) {
        const double* a = P.Arows + (size_t)i * nv;
        double s = 0.0;
        for (int c = 0; c < nv; ++c) s = fma(__ldg(a + c), c == col ? yk : z[c], s);
        double h = __ldg(P.brows + i);
        const int r = i - ne;   // inequality numbering
        if (r >= P.rb0) {
            const int kk = (r - P.rb0) >> 1;
            if (kk < depth) { const double v = (double)((node >> kk) & 1ull); h = ((r - P.rb0) & 1) ? -v : v; }
        }
        const double tol = PPG_FEAS_TOL * (1.0 + fabs(h));
        ok = i < ne ? fabs(s - h) <= tol : s - h <= tol;
    }
    status_out[j] = ok ? PPG_TREE_FEASIBLE : PPG_TREE_UNDECIDED;
    if (!ok) return;
    if (iters_out) iters_out[j] = -1;
    if (point_out)
        for (int c = 0; c < nv; ++c) point_out[(size_t)j * nv + c] = c == col ? yk : z[c];
}

__global__ void k11_tree_children_kernel(const uint64_t* __restrict__ nodes, const long long* __restrict__ idx,
                                         const long long* __restrict__ d_count, long long n_max, int depth,
                                         uint64_t* __restrict__ children, long long* __restrict__ parent_of) {
    const long long cnt = *d_count;
    for (long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x; j < cnt && j < n_max;
         j += (long long)gridDim.x * blockDim.x) {
        const long long p = idx[j];
        const uint64_t v = nodes[p];
        children[2 * j] = v;
        children[2 * j + 1] = v | (1ull << depth);
        parent_of[2 * j] = p;
        parent_of[2 * j + 1] = p;
    }
}

cudaError_t launch_tree_node(const DevTree& P, const uint64_t* nodes, long long n, int depth, uint8_t* status, double* point,
                             int* iters, int skip_done, int sm_count, cudaStream_t st) {
    if (n <= 0) return cudaSuccess;
    const size_t warp_bytes = (size_t)k11_layout(P.rows, P.cols).stride * sizeof(double);
    WarpGrid g;
    const cudaError_t e = warp_grid(k11_tree_node_kernel, warp_bytes, 0, K11_MAX_WARPS, n, sm_count, &g);
    if (e != cudaSuccess) return e;
    k11_tree_node_kernel<<<g.grid, g.warps * 32, g.smem, st>>>(P, nodes, n, depth, status, point, iters, skip_done);
    return cudaGetLastError();
}

cudaError_t launch_tree_inherit(const DevTree& P, const uint64_t* nodes, long long n, int depth, const double* parent_point,
                                const long long* parent_of, uint8_t* status, double* point, int* iters, cudaStream_t st) {
    if (n <= 0) return cudaSuccess;
    if (depth < 1) return cudaErrorInvalidValue;
    const int threads = 128;
    k11_tree_inherit_kernel<<<(unsigned)((n + threads - 1) / threads), threads, 0, st>>>(P, nodes, n, depth, parent_point,
                                                                                         parent_of, status, point, iters);
    return cudaGetLastError();
}

cudaError_t launch_tree_children(const uint64_t* nodes, const long long* idx, const long long* d_count, long long n_max, int depth,
                                 uint64_t* children, long long* parent_of, cudaStream_t st) {
    if (n_max <= 0) return cudaSuccess;
    const int threads = 256;
    long long grid = (n_max + threads - 1) / threads;
    if (grid > 65536) grid = 65536;
    k11_tree_children_kernel<<<(unsigned)grid, threads, 0, st>>>(nodes, idx, d_count, n_max, depth, children, parent_of);
    return cudaGetLastError();
}

}  // namespace ppgpu
