// K9 - batched fixed-parameter LP solves (MPLP_Program.solve_theta / sample_theta_space, verify_solution of an mpLP).
//
// For a fixed theta the reduced LP (host_math.hpp::reduce_program) is  min g(theta)' v  s.t.  At v <= bti + Ft theta,  v free.
// The host exchanged v against np slacks once per program (build_lp_dictionary); per point the kernel
//   1. copies that dictionary into the warp's shared memory with one auxiliary column (Chvatal's x0: every slack row gets
//      s_B = beta - D s_N + x0, the rows of v do not), evaluates beta(theta) and the objective row d(theta) (t + 1 FMAs per
//      entry) and the tolerance of every slack, delta_i = PPG_TLP_TOL (1 + |bti_i + Ft_i theta|);
//   2. Phase 1, when some slack row is below -delta of its slack: x0 enters on the most negative row (lowest row on ties),
//      then the x0 row is minimised; it leaves as soon as it blocks (it is preferred among the rows tied in the ratio
//      test), which ends Phase 1.  At the Phase 1 optimum x0 > delta (of the row it entered on) is infeasible; x0 basic at zero is
//      pivoted out on its largest entry;
//   3. Phase 2 on d(theta) with the x0 column frozen: optimal when no d_j exceeds PPG_TLP_OPT (1 + max |c + H theta|),
//      unbounded when no slack row blocks the entering column.
// Both phases use the rules of lp_core.cuh: Dantzig pricing (lowest column on ties), the Harris ratio test over the slack
// rows only (the rows of v are free: they never block and never leave), the largest pivot among the rows within the Harris
// bound (lowest row on ties), and Bland's rule (lowest variable id) after PPG_BLAND_AFTER degenerate pivots.  Every decision
// depends on the point alone, never on its batch or on the warps per CTA.
//
// Outputs: v from the rows of v, refined against the original rows of the final basis (K9_REFINE passes of
// v += At_N^-1 (bti_N + Ft_N theta - At_N v), At_N^-1 read off the rows of v), x = X0t [1; theta] + Q2 v; lambda_i = -d_j of
// the nonbasic slack i (zero for basic rows), refined the same way against g + At_N' lambda_N = 0; the equality multipliers
// mu = -Pm (c + H theta + A_in' lambda), so that c + H theta + A' dual = 0; the nonbasic slacks as a candidate mask (np rows
// at a vertex); the pivots of both phases and of Phase 1.
//
// One warp per point, the grid strides over points.  Per warp in shared memory: the dictionary (mi + 1 rows incl. the
// objective row, row stride LD = np + 2 rounded up to odd so that lanes walking a column hit distinct banks), the pivot
// row, the tolerances (by slack id), theta, the row / column variable ids and the output staging.  A pivot splits the rows
// over the lanes (each lane updates its rows over all columns); pricing splits the columns, the ratio test the rows; every
// decision is taken on warp-reduced values, so the lanes never diverge.
#include <cmath>

#include "common.cuh"
#include "launch.h"

namespace ppgpu {

constexpr int K9_MAX_WARPS = 16;
constexpr int K9_NONE = 0x7fffffff;
constexpr int K9_REFINE = 2;   // refinement passes of v against the original rows of the optimal basis

struct K9Layout {   // per-warp scratch, in doubles
    int LD, T, P, tol, th, ro, bvar, nvar, mask, stride;
};

__host__ __device__ inline K9Layout k9_layout(int mi, int np, int t, int n, int W) {
    K9Layout o;
    o.LD = (np + 2) | 1;
    int p = 0;
    o.T = p; p += (mi + 1) * o.LD;
    o.P = p; p += o.LD;
    o.tol = p; p += mi;
    o.th = p; p += t;
    o.ro = p; p += n;
    o.bvar = p; p += (mi + 1) / 2;       // ints
    o.nvar = p; p += (np + 2) / 2;       // ints (np + 1 columns)
    o.mask = p; p += W;                  // uint64
    o.stride = p + (p & 1);              // 16-byte aligned warps
    return o;
}

__device__ __forceinline__ void k9_argmin(double& v, int& i) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const double ov = __shfl_xor_sync(0xffffffffu, v, o);
        const int oi = __shfl_xor_sync(0xffffffffu, i, o);
        if (ov < v || (ov == v && oi < i)) { v = ov; i = oi; }
    }
}

__global__ void __launch_bounds__(K9_MAX_WARPS * 32)
k9_theta_lp_kernel(DevProgram P, const double* __restrict__ theta, long long n_points, uint8_t* __restrict__ status_out,
                   double* __restrict__ x_out, double* __restrict__ dual_out, uint64_t* __restrict__ mask_out,
                   int* __restrict__ iters_out) {
    extern __shared__ double k9_smem[];
    const int mi = P.mi, np = P.np, t = P.t, t1 = t + 1, n = P.n, ne = P.ne, Wd = P.W, ld0 = P.lp_ld;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, wpb = blockDim.x >> 5;
    const K9Layout lo = k9_layout(mi, np, t, n, Wd);
    const int LD = lo.LD, nc = np + 1, AUX = mi;   // nonbasic columns 0..np (column np starts as x0); variable id of x0
    double* base = k9_smem + (size_t)warp * lo.stride;
    double* T = base + lo.T;
    double* Pr = base + lo.P;
    double* tolv = base + lo.tol;
    double* th = base + lo.th;
    double* ro = base + lo.ro;
    int* bvar = (int*)(base + lo.bvar);
    int* nvar = (int*)(base + lo.nvar);
    uint64_t* wmask = (uint64_t*)(base + lo.mask);
    double* obj = T + (size_t)mi * LD;
    const double INF = __longlong_as_double(0x7ff0000000000000ll);
    const double QNAN = __longlong_as_double(0x7ff8000000000000ll);

    for (long long pt = (long long)blockIdx.x * wpb + warp; pt < n_points; pt += (long long)gridDim.x * wpb) {
        __syncwarp();
        for (int k = lane; k < t; k += 32) th[k] = theta[pt * t + k];
        for (int k = lane; k < Wd; k += 32) wmask[k] = 0ull;
        // constant entries: row by row, lanes over the columns (coalesced reads of the start dictionary)
        for (int r = 0; r < mi; ++r)
            for (int c = lane; c < np; c += 32) T[(size_t)r * LD + 1 + c] = __ldg(P.lp_D0 + (size_t)r * ld0 + 1 + c);
        __syncwarp();
        for (int r = lane; r < mi; r += 32) {
            const double* src = P.lp_D0 + (size_t)r * ld0;
            double b = __ldg(src);
            for (int k = 0; k < t; ++k) b = fma(-__ldg(src + 1 + np + k), th[k], b);
            const int bv = __ldg(P.lp_bvar + r);
            T[(size_t)r * LD] = b;
            T[(size_t)r * LD + 1 + np] = bv >= 0 ? -1.0 : 0.0;
            bvar[r] = bv;
            // tolerance of slack r on the scale of its own right-hand side bti_r + Ft_r theta (T0 holds -Ft)
            const double* t0 = P.T0 + (size_t)r * P.dc0;
            double h = __ldg(t0);
            for (int k = 0; k < t; ++k) h = fma(-__ldg(t0 + 1 + np + k), th[k], h);
            tolv[r] = PPG_TLP_TOL * (1.0 + fabs(h));
        }
        for (int c = lane; c < np; c += 32) {
            const double* src = P.lp_obj + (size_t)c * t1;
            double d = __ldg(src);
            for (int k = 0; k < t; ++k) d = fma(__ldg(src + 1 + k), th[k], d);
            obj[1 + c] = d;
            nvar[c] = __ldg(P.lp_nvar + c);
        }
        double cmax = 0.0;
        for (int i = lane; i < n; i += 32) {
            double v = __ldg(P.c + i);
            for (int k = 0; k < t; ++k) v = fma(__ldg(P.H + (size_t)i * t + k), th[k], v);
            cmax = fmax(cmax, fabs(v));
        }
        if (lane == 0) { obj[0] = 0.0; obj[1 + np] = 0.0; nvar[np] = AUX; }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) cmax = fmax(cmax, __shfl_xor_sync(0xffffffffu, cmax, o));
        const double opt2 = PPG_TLP_OPT * (1.0 + cmax);
        __syncwarp();

        int it = 0, it1 = 0, status = -1, degen = 0, aux_row = -1;
        double aux_tol = 0.0;   // tolerance of x0: that of the slack it entered on
        bool bland = false;
        // one Gauss-Jordan exchange: basic row l leaves, nonbasic column j enters; false on a non-finite pivot
        auto pivot = [&](int l, int j) -> bool {
            const int cj = 1 + j;
            const double inv = 1.0 / T[(size_t)l * LD + cj];
            if (!isfinite(inv)) return false;
            for (int c = lane; c <= nc; c += 32) Pr[c] = c == cj ? inv : T[(size_t)l * LD + c] * inv;
            __syncwarp();
            for (int r = lane; r <= mi; r += 32) {
                if (r == l) continue;
                double* row = T + (size_t)r * LD;
                const double col = row[cj];
                if (col == 0.0) continue;
                for (int c = 0; c <= nc; ++c) row[c] = fma(-col, Pr[c], row[c]);
                row[cj] = -col * inv;
                if (r < mi && bvar[r] >= 0 && row[0] < 0.0 && row[0] > -(bvar[r] == AUX ? aux_tol : tolv[bvar[r]])) row[0] = 0.0;
            }
            __syncwarp();
            for (int c = lane; c <= nc; c += 32) T[(size_t)l * LD + c] = Pr[c];
            if (lane == 0) { const int b = bvar[l]; bvar[l] = nvar[j]; nvar[j] = b; }
            __syncwarp();
            ++it;
            return true;
        };

        // Phase 1 entry: x0 enters on the most negative slack row beyond its tolerance
        {
            double bv = INF;
            int best = K9_NONE;
            for (int r = lane; r < mi; r += 32) {
                const double v = T[(size_t)r * LD];
                if (bvar[r] >= 0 && v < -tolv[bvar[r]] && v < bv) { bv = v; best = r; }
            }
            k9_argmin(bv, best);
            best = __shfl_sync(0xffffffffu, best, 0);
            if (best != K9_NONE) {
                aux_tol = tolv[bvar[best]];
                if (!pivot(best, np)) status = PPG_TLP_NUMERIC;
                aux_row = best;
                it1 = 1;
            }
        }
        while (status < 0) {
            const bool ph1 = aux_row >= 0;
            const double* orow = ph1 ? T + (size_t)aux_row * LD : obj;
            const double otol = ph1 ? PPG_TLP_OPT : opt2;
            // pricing over the columns: Dantzig (largest d_j, lowest column on ties) or Bland (lowest variable id)
            double key = INF;
            int jc = K9_NONE;
            for (int c = lane; c < nc; c += 32) {
                const double d = orow[1 + c];
                if (nvar[c] == AUX || !(d > otol)) continue;
                const double k = bland ? (double)nvar[c] : -d;
                if (k < key) { key = k; jc = c; }
            }
            k9_argmin(key, jc);
            const int j = __shfl_sync(0xffffffffu, jc, 0);
            if (j == K9_NONE) {
                if (!ph1) { status = PPG_TLP_OPTIMAL; break; }
                if (T[(size_t)aux_row * LD] > aux_tol) { status = PPG_TLP_INFEASIBLE; break; }
                // x0 basic at zero: pivot it out on its largest entry
                double big = -1.0;
                int bc = K9_NONE;
                for (int c = lane; c < nc; c += 32) {
                    const double a = fabs(T[(size_t)aux_row * LD + 1 + c]);
                    if (a > big) { big = a; bc = c; }
                }
                big = -big;
                k9_argmin(big, bc);
                bc = __shfl_sync(0xffffffffu, bc, 0);
                if (!(-big > PPG_TLP_PIV)) { status = PPG_TLP_NUMERIC; break; }
                if (it >= PPG_TLP_MAX_ITER) { status = PPG_TLP_ITERLIM; break; }
                __syncwarp();
                if (lane == 0) T[(size_t)aux_row * LD] = 0.0;
                __syncwarp();
                if (!pivot(aux_row, bc)) { status = PPG_TLP_NUMERIC; break; }
                ++it1;
                aux_row = -1;
                continue;
            }
            if (it >= PPG_TLP_MAX_ITER) { status = PPG_TLP_ITERLIM; break; }
            // Harris ratio test over the slack rows (and x0's row in Phase 1)
            double hb = INF;
            for (int r = lane; r < mi; r += 32) {
                if (bvar[r] < 0) continue;
                const double a = T[(size_t)r * LD + 1 + j];
                if (!(a > PPG_TLP_TINY)) continue;
                const double rhs = fmax(T[(size_t)r * LD], 0.0);
                hb = fmin(hb, (rhs + (bvar[r] == AUX ? aux_tol : tolv[bvar[r]])) / a);
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) hb = fmin(hb, __shfl_xor_sync(0xffffffffu, hb, o));
            if (hb == INF) { status = ph1 ? PPG_TLP_NUMERIC : PPG_TLP_UNBOUNDED; break; }
            // among the rows within the bound: x0's row, else the largest pivot (Bland: lowest variable id), lowest row on ties
            double sel = INF, step = INF;
            int lr = K9_NONE;
            for (int r = lane; r < mi; r += 32) {
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
            if (l == K9_NONE) { status = PPG_TLP_NUMERIC; break; }
            if (step <= PPG_DEGEN_STEP) { if (++degen > PPG_BLAND_AFTER) bland = true; } else degen = 0;
            const bool aux_leaves = l == aux_row;
            if (!pivot(l, j)) { status = PPG_TLP_NUMERIC; break; }
            if (ph1) ++it1;
            if (aux_leaves) aux_row = -1;
        }
        __syncwarp();
        if (status == PPG_TLP_OPTIMAL)
            for (int r = lane; r < mi; r += 32)
                if (!isfinite(T[(size_t)r * LD])) status = PPG_TLP_NUMERIC;
        status = __reduce_max_sync(0xffffffffu, status);
        // nonbasic slacks -> mask (np of them at a vertex; the frozen x0 column is skipped)
        if (lane == 0)
            for (int c = 0; c < nc; ++c)
                if (nvar[c] < AUX) wmask[nvar[c] >> 6] |= 1ull << (nvar[c] & 63);
        __syncwarp();
        if (lane == 0) status_out[pt] = (uint8_t)status;
        if (iters_out && lane == 0) { iters_out[2 * pt] = it; iters_out[2 * pt + 1] = it1; }
        if (mask_out) for (int k = lane; k < Wd; k += 32) mask_out[pt * Wd + k] = wmask[k];
        if (!x_out && !dual_out) continue;
        if (status != PPG_TLP_OPTIMAL) {
            if (x_out) for (int i = lane; i < n; i += 32) x_out[pt * n + i] = QNAN;
            if (dual_out) for (int i = lane; i < P.m; i += 32) dual_out[pt * P.m + i] = QNAN;
            continue;
        }
        // v (staged in the pivot row) and x
        for (int r = lane; r < mi; r += 32)
            if (bvar[r] < 0) Pr[-1 - bvar[r]] = T[(size_t)r * LD];
        __syncwarp();
        // the rows of v carry the rounding of every pivot (entries of 1e7 box rows next to rows near 1): refine v against the
        // original rows of the final basis, At_N v = bti_N + Ft_N theta, with D_v = At_N^-1 from the same dictionary
        for (int pass = 0; pass < K9_REFINE; ++pass) {
            for (int c = lane; c < nc; c += 32) {
                const int s = nvar[c];
                if (s >= AUX) continue;
                const double* t0 = P.T0 + (size_t)s * P.dc0;
                double h = __ldg(t0);
                for (int k = 0; k < t; ++k) h = fma(-__ldg(t0 + 1 + np + k), th[k], h);
                for (int j = 0; j < np; ++j) h = fma(-__ldg(t0 + 1 + j), Pr[j], h);
                tolv[s] = h;   // residual slack of the nonbasic row s (tolv is free now)
            }
            __syncwarp();
            for (int r = lane; r < mi; r += 32) {
                if (bvar[r] >= 0) continue;
                const double* row = T + (size_t)r * LD;
                double dv = 0.0;
                for (int c = 0; c < nc; ++c)
                    if (nvar[c] < AUX) dv = fma(row[1 + c], tolv[nvar[c]], dv);
                ro[-1 - bvar[r]] = dv;
            }
            __syncwarp();
            for (int j = lane; j < np; j += 32) Pr[j] += ro[j];
            __syncwarp();
        }
        if (x_out)
            for (int i = lane; i < n; i += 32) {
                const double* xr = P.X0t + (size_t)i * t1;
                double v = __ldg(xr);
                for (int k = 0; k < t; ++k) v = fma(__ldg(xr + 1 + k), th[k], v);
                for (int c = 0; c < np; ++c) v = fma(__ldg(P.Q2 + (size_t)i * np + c), Pr[c], v);
                x_out[pt * n + i] = v;
            }
        if (!dual_out) continue;
        __syncwarp();
        // lambda of the nonbasic slacks, scattered over the rows (tolv is free now)
        for (int r = lane; r < mi; r += 32) tolv[r] = 0.0;
        __syncwarp();
        for (int c = lane; c < nc; c += 32)
            if (nvar[c] < AUX) tolv[nvar[c]] = -obj[1 + c];
        // ... refined as v is: g + At_N' lambda_N = 0 with g = Q2' (c + H theta), lambda_N -= At_N^-T (g + At_N' lambda_N)
        for (int i = lane; i < n; i += 32) {
            double v = __ldg(P.c + i);
            for (int k = 0; k < t; ++k) v = fma(__ldg(P.H + (size_t)i * t + k), th[k], v);
            ro[i] = v;
        }
        __syncwarp();
        for (int j = lane; j < np; j += 32) {
            double v = 0.0;
            for (int i = 0; i < n; ++i) v = fma(__ldg(P.Q2 + (size_t)i * np + j), ro[i], v);
            Pr[j] = v;   // g (v is no longer needed)
        }
        __syncwarp();
        for (int pass = 0; pass < K9_REFINE; ++pass) {
            for (int j = lane; j < np; j += 32) {
                double v = Pr[j];
                for (int c = 0; c < nc; ++c) {
                    const int s = nvar[c];
                    if (s < AUX) v = fma(__ldg(P.T0 + (size_t)s * P.dc0 + 1 + j), tolv[s], v);
                }
                ro[j] = v;   // stationarity residual in v
            }
            __syncwarp();
            double dl[3] = {0.0, 0.0, 0.0};   // nc <= 65 columns: at most 3 per lane
            for (int r = 0; r < mi; ++r) {
                if (bvar[r] >= 0) continue;
                const double rho = ro[-1 - bvar[r]];
                for (int q = 0; q < 3; ++q) {
                    const int c = lane + 32 * q;
                    if (c < nc) dl[q] = fma(T[(size_t)r * LD + 1 + c], rho, dl[q]);
                }
            }
            __syncwarp();
            for (int q = 0; q < 3; ++q) {
                const int c = lane + 32 * q;
                if (c < nc && nvar[c] < AUX) tolv[nvar[c]] -= dl[q];
            }
            __syncwarp();
        }
        for (int r = lane; r < mi; r += 32) dual_out[pt * P.m + ne + r] = tolv[r];
        if (ne == 0) continue;
        for (int i = lane; i < n; i += 32) {
            double v = __ldg(P.c + i);
            for (int k = 0; k < t; ++k) v = fma(__ldg(P.H + (size_t)i * t + k), th[k], v);
            for (int c = 0; c < nc; ++c) {
                const int s = nvar[c];
                if (s < AUX) v = fma(__ldg(P.A + (size_t)(ne + s) * n + i), tolv[s], v);
            }
            ro[i] = v;
        }
        __syncwarp();
        for (int e = lane; e < ne; e += 32) {
            double v = 0.0;
            for (int i = 0; i < n; ++i) v = fma(__ldg(P.Pm + (size_t)e * n + i), ro[i], v);
            dual_out[pt * P.m + e] = -v;
        }
    }
}

cudaError_t launch_theta_lp(const DevProgram& P, const double* theta, long long n_points, uint8_t* status, double* x,
                            double* dual, uint64_t* mask, int* iters, int sm_count, cudaStream_t st) {
    if (n_points <= 0) return cudaSuccess;
    if (P.is_qp || !P.lp_ok || P.np > 64) return cudaErrorInvalidValue;
    int dev = 0, lim = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&lim, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
    if (e != cudaSuccess) return e;
    cudaFuncAttributes fa;
    if ((e = cudaFuncGetAttributes(&fa, k9_theta_lp_kernel)) != cudaSuccess) return e;
    const size_t warp_bytes = (size_t)k9_layout(P.mi, P.np, P.t, P.n, P.W).stride * sizeof(double);
    const size_t avail = (size_t)lim - fa.sharedSizeBytes;   // static shared memory counts against the same limit
    int wpb = (int)(avail / warp_bytes);
    if (wpb > K9_MAX_WARPS) wpb = K9_MAX_WARPS;
    if (wpb < 1) return cudaErrorInvalidValue;
    const size_t smem = (size_t)wpb * warp_bytes;
    if ((e = fit_smem(k9_theta_lp_kernel, smem)) != cudaSuccess) return e;
    int per_sm = 0;
    if ((e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k9_theta_lp_kernel, wpb * 32, smem)) != cudaSuccess) return e;
    if (per_sm < 1) per_sm = 1;
    long long grid = (n_points + wpb - 1) / wpb;
    const long long cap = (long long)sm_count * per_sm;
    if (grid > cap) grid = cap;
    k9_theta_lp_kernel<<<(unsigned)grid, wpb * 32, smem, st>>>(P, theta, n_points, status, x, dual, mask, iters);
    return cudaGetLastError();
}

}  // namespace ppgpu
