// K11 - the relaxation tree of a mixed-integer program (mpmiqp_enumeration's screen of the binary assignments).
//
// A node at depth d fixes y_0..y_{d-1}; it is feasible iff the LP relaxation of the lifted system (host_math.hpp::TreeProgram:
// z = (x, theta), the program's rows, Theta's rows and two bound rows per binary) has a point within PPG_FEAS_TOL.  The
// dictionary entries are the same for every node; only the right-hand side depends on the node's bounds.
//
// k11_tree_node_kernel, one warp per node, grid-stride:
//   1. copies the dictionary into the warp's shared memory with one auxiliary column (Chvatal's x0: every slack row gets
//      s_B = beta - D s_N + x0, the rows of v do not), evaluates beta(node) = beta0 + sum_{k<d} Dbnd[:, 2k + y_k] and the
//      Harris relaxation of every slack, PPG_TREE_HARRIS (1 + |h_i|) with h_i the row's right-hand side at the node;
//   2. Phase 1 only: when some slack row is below its relaxation, x0 enters on the most negative row (lowest row on ties),
//      then the x0 row is minimised.  Feasible as soon as x0 leaves (it is preferred among the rows tied in the ratio test)
//      or when the minimum is at most PPG_TREE_AUX; infeasible when it is larger.
//   K9's rules (k9_theta_lp.cu): Dantzig pricing (lowest column on ties), the Harris ratio test over the slack rows only (the
//   rows of v are free: they never block and never leave), the largest pivot among the rows within the Harris bound (lowest
//   row on ties), and Bland's rule (lowest variable id) after PPG_BLAND_AFTER degenerate pivots.  Every decision depends on
//   the node alone, never on its batch or on the warps per CTA.
//   Outputs: a status byte, the pivot count and, when asked for, the point z = z0 + Q2 v of the final dictionary.
// k11_tree_inherit_kernel, one thread per node: the parent's point with the newly fixed binary snapped to the node's value is
//   checked against every lifted row at the node's bounds with the verdict's tolerance; when it holds, the node is feasible
//   without an LP and inherits that point.  It never decides infeasibility.
// k11_tree_children_kernel, one thread per selected (feasible) node: children in parent order, y_d = 0 before y_d = 1, so
//   the leaves come out in lexicographic order of (y_0, y_1, ...).
#include <cmath>

#include "common.cuh"
#include "launch.h"

namespace ppgpu {

constexpr int K11_MAX_WARPS = 16;
constexpr int K11_NONE = 0x7fffffff;

struct K11Layout {   // per-warp scratch, in doubles
    int LD, T, P, tol, bvar, nvar, stride;
};

__host__ __device__ inline K11Layout k11_layout(int rows, int cols) {
    K11Layout o;
    o.LD = (cols + 2) | 1;   // [beta | cols | x0], odd so that lanes walking a column hit distinct banks
    int p = 0;
    o.T = p; p += rows * o.LD;
    o.P = p; p += o.LD;
    o.tol = p; p += rows;
    o.bvar = p; p += (rows + 1) / 2;     // ints
    o.nvar = p; p += (cols + 2) / 2;     // ints (cols + 1 columns)
    o.stride = p + (p & 1);              // 16-byte aligned warps
    return o;
}

__device__ __forceinline__ void k11_argmin(double& v, int& i) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const double ov = __shfl_xor_sync(0xffffffffu, v, o);
        const int oi = __shfl_xor_sync(0xffffffffu, i, o);
        if (ov < v || (ov == v && oi < i)) { v = ov; i = oi; }
    }
}

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
    const K11Layout lo = k11_layout(rows, cols);
    const int LD = lo.LD, nc = cols + 1, AUX = rows;   // nonbasic columns 0..cols (column cols starts as x0); x0's id
    double* base = k11_smem + (size_t)warp * lo.stride;
    double* T = base + lo.T;
    double* Pr = base + lo.P;
    double* tolv = base + lo.tol;
    int* bvar = (int*)(base + lo.bvar);
    int* nvar = (int*)(base + lo.nvar);
    const double INF = __longlong_as_double(0x7ff0000000000000ll);
    const double QNAN = __longlong_as_double(0x7ff8000000000000ll);
    const double aux_tol = PPG_TREE_AUX;

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

        int it = 0, status = -1, degen = 0, aux_row = -1;
        bool bland = false;
        // one Gauss-Jordan exchange: basic row l leaves, nonbasic column j enters; false on a non-finite pivot
        auto pivot = [&](int l, int j) -> bool {
            const int cj = 1 + j;
            const double inv = 1.0 / T[(size_t)l * LD + cj];
            if (!isfinite(inv)) return false;
            for (int c = lane; c <= nc; c += 32) Pr[c] = c == cj ? inv : T[(size_t)l * LD + c] * inv;
            __syncwarp();
            for (int r = lane; r < rows; r += 32) {
                if (r == l) continue;
                double* row = T + (size_t)r * LD;
                const double col = row[cj];
                if (col == 0.0) continue;
                for (int c = 0; c <= nc; ++c) row[c] = fma(-col, Pr[c], row[c]);
                row[cj] = -col * inv;
                if (bvar[r] >= 0 && row[0] < 0.0 && row[0] > -(bvar[r] == AUX ? aux_tol : tolv[bvar[r]])) row[0] = 0.0;
            }
            __syncwarp();
            for (int c = lane; c <= nc; c += 32) T[(size_t)l * LD + c] = Pr[c];
            if (lane == 0) { const int b = bvar[l]; bvar[l] = nvar[j]; nvar[j] = b; }
            __syncwarp();
            ++it;
            return true;
        };

        // Phase 1 entry: x0 enters on the most negative slack row beyond its relaxation
        {
            double bv = INF;
            int best = K11_NONE;
            for (int r = lane; r < rows; r += 32) {
                const double v = T[(size_t)r * LD];
                if (bvar[r] >= 0 && v < -tolv[bvar[r]] && v < bv) { bv = v; best = r; }
            }
            k11_argmin(bv, best);
            best = __shfl_sync(0xffffffffu, best, 0);
            if (best == K11_NONE) status = PPG_TREE_FEASIBLE;
            else if (!pivot(best, cols)) status = PPG_TLP_NUMERIC;
            else aux_row = best;
        }
        while (status < 0) {
            const double* orow = T + (size_t)aux_row * LD;
            // pricing over the columns: Dantzig (largest d_j, lowest column on ties) or Bland (lowest variable id)
            double key = INF;
            int jc = K11_NONE;
            for (int c = lane; c < nc; c += 32) {
                const double d = orow[1 + c];
                if (!(d > PPG_TLP_OPT)) continue;
                const double k = bland ? (double)nvar[c] : -d;
                if (k < key) { key = k; jc = c; }
            }
            k11_argmin(key, jc);
            const int j = __shfl_sync(0xffffffffu, jc, 0);
            if (j == K11_NONE) { status = orow[0] > aux_tol ? PPG_TREE_INFEASIBLE : PPG_TREE_FEASIBLE; break; }
            if (it >= PPG_TLP_MAX_ITER) { status = PPG_TLP_ITERLIM; break; }
            // Harris ratio test over the slack rows and x0's row
            double hb = INF;
            for (int r = lane; r < rows; r += 32) {
                if (bvar[r] < 0) continue;
                const double a = T[(size_t)r * LD + 1 + j];
                if (!(a > PPG_TLP_TINY)) continue;
                const double rhs = fmax(T[(size_t)r * LD], 0.0);
                hb = fmin(hb, (rhs + (bvar[r] == AUX ? aux_tol : tolv[bvar[r]])) / a);
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) hb = fmin(hb, __shfl_xor_sync(0xffffffffu, hb, o));
            if (hb == INF) { status = PPG_TLP_NUMERIC; break; }   // x0's row blocks a column that decreases it
            // among the rows within the bound: x0's row, else the largest pivot (Bland: lowest variable id), lowest row on ties
            double sel = INF, step = INF;
            int lr = K11_NONE;
            for (int r = lane; r < rows; r += 32) {
                if (bvar[r] < 0) continue;
                const double a = T[(size_t)r * LD + 1 + j];
                if (!(a > PPG_TLP_TINY)) continue;
                const double rat = fmax(T[(size_t)r * LD], 0.0) / a;
                if (!(rat <= hb)) continue;
                const double k = r == aux_row ? -INF : (bland ? (double)bvar[r] : -a);
                if (k < sel) { sel = k; lr = r; step = rat; }
            }
            {
                double s2 = step;
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) {
                    const double ov = __shfl_xor_sync(0xffffffffu, sel, o);
                    const int oi = __shfl_xor_sync(0xffffffffu, lr, o);
                    const double os = __shfl_xor_sync(0xffffffffu, s2, o);
                    if (ov < sel || (ov == sel && oi < lr)) { sel = ov; lr = oi; s2 = os; }
                }
                step = __shfl_sync(0xffffffffu, s2, 0);
            }
            const int l = __shfl_sync(0xffffffffu, lr, 0);
            if (l == K11_NONE) { status = PPG_TLP_NUMERIC; break; }
            if (step <= PPG_DEGEN_STEP) { if (++degen > PPG_BLAND_AFTER) bland = true; } else degen = 0;
            const bool aux_leaves = l == aux_row;
            if (!pivot(l, j)) { status = PPG_TLP_NUMERIC; break; }
            if (aux_leaves) { status = PPG_TREE_FEASIBLE; break; }
        }
        __syncwarp();
        if (status == PPG_TREE_FEASIBLE)
            for (int r = lane; r < rows; r += 32)
                if (!isfinite(T[(size_t)r * LD])) status = PPG_TLP_NUMERIC;
        status = __reduce_max_sync(0xffffffffu, status);
        if (lane == 0) status_out[pt] = (uint8_t)status;
        if (iters_out && lane == 0) iters_out[pt] = it;
        if (!point_out) continue;
        if (status != PPG_TREE_FEASIBLE) {
            for (int i = lane; i < nv; i += 32) point_out[pt * nv + i] = QNAN;
            continue;
        }
        // v from its rows (staged in the pivot row), z = z0 + Q2 v
        for (int r = lane; r < rows; r += 32)
            if (bvar[r] < 0) Pr[-1 - bvar[r]] = T[(size_t)r * LD];
        __syncwarp();
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
    int dev = 0, lim = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&lim, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
    if (e != cudaSuccess) return e;
    cudaFuncAttributes fa;
    if ((e = cudaFuncGetAttributes(&fa, k11_tree_node_kernel)) != cudaSuccess) return e;
    const size_t warp_bytes = (size_t)k11_layout(P.rows, P.cols).stride * sizeof(double);
    const size_t avail = (size_t)lim - fa.sharedSizeBytes;   // static shared memory counts against the same limit
    int wpb = (int)(avail / warp_bytes);
    if (wpb > K11_MAX_WARPS) wpb = K11_MAX_WARPS;
    if (wpb < 1) return cudaErrorInvalidValue;
    const size_t smem = (size_t)wpb * warp_bytes;
    if ((e = fit_smem(k11_tree_node_kernel, smem)) != cudaSuccess) return e;
    int per_sm = 0;
    if ((e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k11_tree_node_kernel, wpb * 32, smem)) != cudaSuccess) return e;
    if (per_sm < 1) per_sm = 1;
    long long grid = (n + wpb - 1) / wpb;
    const long long cap = (long long)sm_count * per_sm;
    if (grid > cap) grid = cap;
    k11_tree_node_kernel<<<(unsigned)grid, wpb * 32, smem, st>>>(P, nodes, n, depth, status, point, iters, skip_done);
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
