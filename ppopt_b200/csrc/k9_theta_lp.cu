// K9 - batched fixed-parameter LP solves (MPLP_Program.solve_theta / sample_theta_space, verify_solution of an mpLP).
//
// For a fixed theta the reduced LP (host_math.hpp::reduce_program) is  min g(theta)' v  s.t.  At v <= bti + Ft theta,  v free.
// The host exchanged v against np slacks once per program (build_lp_dictionary); per point the kernel
//   1. copies that dictionary into the warp's shared memory with the auxiliary column x0 of warp_dict.cuh and the objective
//      row below the mi rows, evaluates beta(theta) and the objective row d(theta) (t + 1 FMAs per entry) and the tolerance
//      of every slack, delta_i = PPG_TLP_TOL (1 + |bti_i + Ft_i theta|);
//   2. Phase 1, when some slack row is below -delta of its slack: x0 enters (its tolerance is that of the slack it entered
//      on), then the x0 row is minimised; it leaves as soon as it blocks, which ends Phase 1.  At the Phase 1 optimum
//      x0 > its tolerance is infeasible; x0 basic at zero is pivoted out on its largest entry;
//   3. Phase 2 on d(theta) with the x0 column frozen: optimal when no d_j exceeds PPG_TLP_OPT (1 + max |c + H theta|),
//      unbounded when no slack row blocks the entering column.
// Both phases follow the rules of warp_dict.cuh.
//
// Outputs: v from the rows of v, refined against the original rows of the final basis (K9_REFINE passes of
// v += At_N^-1 (bti_N + Ft_N theta - At_N v), At_N^-1 read off the rows of v), x = X0t [1; theta] + Q2 v; lambda_i = -d_j of
// the nonbasic slack i (zero for basic rows), refined the same way against g + At_N' lambda_N = 0; the equality multipliers
// mu = -Pm (c + H theta + A_in' lambda), so that c + H theta + A' dual = 0; the nonbasic slacks as a candidate mask (np rows
// at a vertex); the pivots of both phases and of Phase 1.
//
// One warp per point, the grid strides over points.  Per warp in shared memory: the dictionary of warp_dict.cuh (mi + 1
// rows incl. the objective row), then theta, a row of n doubles for the refinement and the output staging, and the mask.
//
// Pair mode (PairArgs, an mpMILP at fixed binary assignments; a separate instantiation): the assignment's terms
// [d_y | f_y | x_y] enter as beta = beta0 - Dth theta - d_y, the slack scale and refinement right-hand side
// bti + Ft theta + f_y, and x = X0t [1; theta] + x_y + Q2 v; the objective row does not depend on y; obj receives
// (c + H theta)' x per pair.
#include <cmath>

#include "common.cuh"
#include "launch.h"
#include "warp_dict.cuh"

namespace ppgpu {

constexpr int K9_MAX_WARPS = 16;
constexpr int K9_REFINE = 2;   // refinement passes of v against the original rows of the optimal basis

// the dictionary, then theta (t), a row of n and the mask (W uint64)
__host__ __device__ inline WarpDictLayout k9_layout(int mi, int np, int t, int n, int W) {
    return warp_dict_layout(mi, mi + 1, np, t + n + W);
}

// PAIRS: the pair mode of PairArgs (a separate instantiation: the point mode's code is the one without it)
template <bool PAIRS>
__global__ void __launch_bounds__(K9_MAX_WARPS * 32)
k9_theta_lp_kernel(DevProgram P, const double* __restrict__ theta, long long n_points, uint8_t* __restrict__ status_out,
                   double* __restrict__ x_out, double* __restrict__ dual_out, uint64_t* __restrict__ mask_out,
                   int* __restrict__ iters_out, PairArgs pa) {
    extern __shared__ double k9_smem[];
    const int mi = P.mi, np = P.np, t = P.t, t1 = t + 1, n = P.n, ne = P.ne, Wd = P.W, ld0 = P.lp_ld;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, wpb = blockDim.x >> 5;
    const WarpDictLayout lo = k9_layout(mi, np, t, n, Wd);
    const int LD = lo.LD, nc = np + 1, AUX = mi;   // nonbasic columns 0..np (column np starts as x0); variable id of x0
    double* base = k9_smem + (size_t)warp * lo.stride;
    double* T = base + lo.T;
    double* Pr = base + lo.P;
    double* tolv = base + lo.tol;
    int* bvar = (int*)(base + lo.bvar);
    int* nvar = (int*)(base + lo.nvar);
    double* th = base + lo.extra;
    double* ro = th + t;
    uint64_t* wmask = (uint64_t*)(ro + n);
    double* obj = T + (size_t)mi * LD;
    const double QNAN = __longlong_as_double(0x7ff8000000000000ll);

    for (long long pt = (long long)blockIdx.x * wpb + warp; pt < n_points; pt += (long long)gridDim.x * wpb) {
        __syncwarp();
        const double* oy = nullptr;   // the pair's assignment terms [d_y | f_y | x_y]
        if (PAIRS) {
            const long long tp = pa.pairs[2 * pt];
            oy = pa.off + (long long)pa.pairs[2 * pt + 1] * pa.off_ld;
            for (int k = lane; k < t; k += 32) th[k] = theta[tp * t + k];
        } else {
            for (int k = lane; k < t; k += 32) th[k] = theta[pt * t + k];
        }
        for (int k = lane; k < Wd; k += 32) wmask[k] = 0ull;
        // constant entries: row by row, lanes over the columns (coalesced reads of the start dictionary)
        for (int r = 0; r < mi; ++r)
            for (int c = lane; c < np; c += 32) T[(size_t)r * LD + 1 + c] = __ldg(P.lp_D0 + (size_t)r * ld0 + 1 + c);
        __syncwarp();
        for (int r = lane; r < mi; r += 32) {
            const double* src = P.lp_D0 + (size_t)r * ld0;
            double b = __ldg(src);
            for (int k = 0; k < t; ++k) b = fma(-__ldg(src + 1 + np + k), th[k], b);
            if (PAIRS) b -= oy[r];
            const int bv = __ldg(P.lp_bvar + r);
            T[(size_t)r * LD] = b;
            T[(size_t)r * LD + 1 + np] = bv >= 0 ? -1.0 : 0.0;
            bvar[r] = bv;
            // tolerance of slack r on the scale of its own right-hand side bti_r + Ft_r theta (T0 holds -Ft)
            const double* t0 = P.T0 + (size_t)r * P.dc0;
            double h = __ldg(t0);
            for (int k = 0; k < t; ++k) h = fma(-__ldg(t0 + 1 + np + k), th[k], h);
            if (PAIRS) h += oy[mi + r];
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

        // x0's tolerance is that of the slack it enters on
        WarpDict wd{T, Pr, tolv, bvar, nvar, LD, mi, mi + 1, nc, lane, 0.0};
        int it1 = 0, status = -1, aux_row = -1;
        const int entry = wd.x0_row();
        if (entry != WD_NONE) {
            wd.aux_tol = tolv[bvar[entry]];
            if (!wd.pivot(entry, np)) status = PPG_TLP_NUMERIC;
            aux_row = entry;
            it1 = 1;
        }
        while (status < 0) {
            const bool ph1 = aux_row >= 0;
            const int j = wd.price(ph1 ? T + (size_t)aux_row * LD : obj, ph1 ? PPG_TLP_OPT : opt2);
            if (j == WD_NONE) {
                if (!ph1) { status = PPG_TLP_OPTIMAL; break; }
                if (wd.rhs(aux_row) > wd.aux_tol) { status = PPG_TLP_INFEASIBLE; break; }
                // x0 basic at zero: pivot it out on its largest entry
                double big = -1.0;
                int bc = WD_NONE;
                for (int c = lane; c < nc; c += 32) {
                    const double a = fabs(T[(size_t)aux_row * LD + 1 + c]);
                    if (a > big) { big = a; bc = c; }
                }
                big = -big;
                warp_argmin(big, bc);
                bc = __shfl_sync(PPG_FULL, bc, 0);
                if (!(-big > PPG_TLP_PIV)) { status = PPG_TLP_NUMERIC; break; }
                if (wd.it >= PPG_TLP_MAX_ITER) { status = PPG_TLP_ITERLIM; break; }
                __syncwarp();
                if (lane == 0) T[(size_t)aux_row * LD] = 0.0;
                __syncwarp();
                if (!wd.pivot(aux_row, bc)) { status = PPG_TLP_NUMERIC; break; }
                ++it1;
                aux_row = -1;
                continue;
            }
            if (wd.it >= PPG_TLP_MAX_ITER) { status = PPG_TLP_ITERLIM; break; }
            const WarpDict::Ratio q = wd.ratio(j, aux_row);
            if (!q.blocked) { status = ph1 ? PPG_TLP_NUMERIC : PPG_TLP_UNBOUNDED; break; }
            if (q.row == WD_NONE) { status = PPG_TLP_NUMERIC; break; }
            wd.count_step(q.step);
            if (!wd.pivot(q.row, j)) { status = PPG_TLP_NUMERIC; break; }
            if (ph1) ++it1;
            if (q.row == aux_row) aux_row = -1;
        }
        status = wd.settle(status, PPG_TLP_OPTIMAL);
        // nonbasic slacks -> mask (np of them at a vertex; the frozen x0 column is skipped)
        if (lane == 0)
            for (int c = 0; c < nc; ++c)
                if (nvar[c] < AUX) wmask[nvar[c] >> 6] |= 1ull << (nvar[c] & 63);
        __syncwarp();
        if (lane == 0) status_out[pt] = (uint8_t)status;
        if (iters_out && lane == 0) { iters_out[2 * pt] = wd.it; iters_out[2 * pt + 1] = it1; }
        if (mask_out) for (int k = lane; k < Wd; k += 32) mask_out[pt * Wd + k] = wmask[k];
        const bool want_obj = PAIRS && pa.obj;
        if (!x_out && !dual_out && !want_obj) continue;
        if (status != PPG_TLP_OPTIMAL) {
            if (x_out) for (int i = lane; i < n; i += 32) x_out[pt * n + i] = QNAN;
            if (dual_out) for (int i = lane; i < P.m; i += 32) dual_out[pt * P.m + i] = QNAN;
            if (want_obj && lane == 0) pa.obj[pt] = QNAN;
            continue;
        }
        // v (staged in the pivot row) and x
        wd.stage_v();
        // the rows of v carry the rounding of every pivot (entries of 1e7 box rows next to rows near 1): refine v against the
        // original rows of the final basis, At_N v = bti_N + Ft_N theta, with D_v = At_N^-1 from the same dictionary
        for (int pass = 0; pass < K9_REFINE; ++pass) {
            for (int c = lane; c < nc; c += 32) {
                const int s = nvar[c];
                if (s >= AUX) continue;
                const double* t0 = P.T0 + (size_t)s * P.dc0;
                double h = __ldg(t0);
                for (int k = 0; k < t; ++k) h = fma(-__ldg(t0 + 1 + np + k), th[k], h);
                if (PAIRS) h += oy[mi + s];
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
        if (x_out || want_obj) {
            double acc = 0.0;   // (c + H theta)' x of the pair (an mpMILP's objective row does not depend on y)
            for (int i = lane; i < n; i += 32) {
                const double* xr = P.X0t + (size_t)i * t1;
                double v = __ldg(xr);
                for (int k = 0; k < t; ++k) v = fma(__ldg(xr + 1 + k), th[k], v);
                if (PAIRS) v += oy[2 * mi + i];
                for (int c = 0; c < np; ++c) v = fma(__ldg(P.Q2 + (size_t)i * np + c), Pr[c], v);
                if (x_out) x_out[pt * n + i] = v;
                if (want_obj) {
                    double g = __ldg(P.c + i);
                    for (int k = 0; k < t; ++k) g = fma(__ldg(P.H + (size_t)i * t + k), th[k], g);
                    acc = fma(g, v, acc);
                }
            }
            if (want_obj) {
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
                if (lane == 0) pa.obj[pt] = acc;
            }
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

template <bool PAIRS>
static cudaError_t launch_k9(const DevProgram& P, const double* theta, const PairArgs& pa, long long n_points, uint8_t* status,
                             double* x, double* dual, uint64_t* mask, int* iters, int sm_count, cudaStream_t st) {
    if (n_points <= 0) return cudaSuccess;
    if (P.is_qp || !P.lp_ok || P.np > 64) return cudaErrorInvalidValue;
    const size_t warp_bytes = (size_t)k9_layout(P.mi, P.np, P.t, P.n, P.W).stride * sizeof(double);
    WarpGrid g;
    const cudaError_t e = warp_grid(k9_theta_lp_kernel<PAIRS>, warp_bytes, 0, K9_MAX_WARPS, n_points, sm_count, &g);
    if (e != cudaSuccess) return e;
    k9_theta_lp_kernel<PAIRS><<<g.grid, g.warps * 32, g.smem, st>>>(P, theta, n_points, status, x, dual, mask, iters, pa);
    return cudaGetLastError();
}

cudaError_t launch_theta_lp(const DevProgram& P, const double* theta, long long n_points, uint8_t* status, double* x,
                            double* dual, uint64_t* mask, int* iters, int sm_count, cudaStream_t st) {
    return launch_k9<false>(P, theta, PairArgs{nullptr, nullptr, 0, nullptr}, n_points, status, x, dual, mask, iters, sm_count, st);
}

cudaError_t launch_theta_lp_pairs(const DevProgram& P, const double* theta, const PairArgs& pa, long long n_pairs, uint8_t* status,
                                  double* x, double* dual, uint64_t* mask, int* iters, int sm_count, cudaStream_t st) {
    if (!pa.pairs || !pa.off) return cudaErrorInvalidValue;
    return launch_k9<true>(P, theta, pa, n_pairs, status, x, dual, mask, iters, sm_count, st);
}

}  // namespace ppgpu
