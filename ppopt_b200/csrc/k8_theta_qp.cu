// K8 - batched fixed-parameter QP solves (MPQP_Program.solve_theta / sample_theta_space, verify_solution of a solution).
//
// For a fixed theta the dual of the reduced QP (host_math.hpp::reduce_program) is the LCP
//     w = G lambda + V [1; theta] >= 0,   lambda >= 0,   lambda' w = 0        (w: slacks of the inequality rows)
// solved by a dual active-set iteration (Goldfarb-Idnani on the dual, the class of DAQP):
//   1. lambda = 0, W empty;
//   2. of the rows outside W violated beyond their tolerance (w_r < -PPG_QP_TOL (1 + |w_r(lambda = 0)|)) the most negative
//      slack w_j enters (lowest row on ties); none: optimal;
//   3. direction from the Cholesky factor L of G_WW:  L l = G_Wj,  L' d = -l,  curvature z = G_jj - |l|^2;
//   4. full step s = -w_j / z (z > PPG_QP_CURV G_jj) or a partial step to the first multiplier of W that reaches zero
//      (d_i < -PPG_QP_DTOL, lowest row on ties), which leaves W while j stays pending; neither: infeasible.
// An add appends the row [l, sqrt(z)] to L; a drop shifts the rows below up without the dropped column and gives the
// trailing block a rank-one update with that column.  The primal point is x = Xp [1; theta] - K lambda, the equality
// multipliers mu = -Pm (Q x + H theta + c + A_in' lambda).  tests/twin_theta_qp.cpp restates the iteration.
//
// One warp per point, the grid strides over points.  G (mi x mi) is staged once per CTA in shared memory when it fits
// next to four warps' scratch, else read through L1/L2.  Per warp in shared memory: w, the per-row tolerances, lambda_W,
// W, L (packed lower triangle), three vectors of np and the output staging.  Lanes split the update
// w += s (G[:,j] + G[:,W] d) (mi x (|W| + 1) FMA per step, rows of G read contiguously: G is symmetric) and the columns of
// the triangular solves; every decision is taken on values broadcast from lane 0, so the lanes never diverge.
#include <cmath>

#include "common.cuh"
#include "launch.h"

namespace ppgpu {

constexpr int K8_MAX_WARPS = 16;

__device__ __forceinline__ int k8_tri(int r, int c) { return r * (r + 1) / 2 + c; }

struct K8Layout {   // per-warp scratch, in doubles
    int w, tol, lam, g, d, xv, L, th, xo, ro, widx, mask, stride;
};

__host__ __device__ inline K8Layout k8_layout(int mi, int np, int t, int n, int W) {
    K8Layout o;
    int p = 0;
    o.w = p; p += mi;
    o.tol = p; p += mi;
    o.lam = p; p += np;
    o.g = p; p += np;
    o.d = p; p += np;
    o.xv = p; p += np;
    o.L = p; p += np * (np + 1) / 2;
    o.th = p; p += t;
    o.xo = p; p += n;
    o.ro = p; p += n;
    o.widx = p; p += (np + 1) / 2;   // ints
    o.mask = p; p += W;              // uint64
    o.stride = p + (p & 1);          // 16-byte aligned warps
    return o;
}

__global__ void __launch_bounds__(K8_MAX_WARPS * 32)
k8_theta_qp_kernel(DevProgram P, const double* __restrict__ theta, long long n_points, int stage_g, uint8_t* __restrict__ status_out,
                   double* __restrict__ x_out, double* __restrict__ dual_out, uint64_t* __restrict__ mask_out,
                   int* __restrict__ iters_out) {
    extern __shared__ double k8_smem[];
    const int mi = P.mi, np = P.np, t = P.t, t1 = t + 1, n = P.n, ne = P.ne, Wd = P.W;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, wpb = blockDim.x >> 5;
    const K8Layout lo = k8_layout(mi, np, t, n, Wd);
    const double* G = P.G;
    double* base = k8_smem;
    if (stage_g) {
        for (int i = threadIdx.x; i < mi * mi; i += blockDim.x) k8_smem[i] = P.G[i];
        __syncthreads();
        G = k8_smem;
        base += ((size_t)mi * mi + 1) & ~(size_t)1;
    }
    base += (size_t)warp * lo.stride;
    double* w = base + lo.w;
    double* tolv = base + lo.tol;
    double* lam = base + lo.lam;
    double* g = base + lo.g;
    double* d = base + lo.d;
    double* xv = base + lo.xv;
    double* L = base + lo.L;
    double* th = base + lo.th;
    double* xo = base + lo.xo;
    double* ro = base + lo.ro;
    int* widx = (int*)(base + lo.widx);
    uint64_t* wmask = (uint64_t*)(base + lo.mask);
    const double INF = __longlong_as_double(0x7ff0000000000000ll);
    const double QNAN = __longlong_as_double(0x7ff8000000000000ll);

    for (long long pt = (long long)blockIdx.x * wpb + warp; pt < n_points; pt += (long long)gridDim.x * wpb) {
        __syncwarp();
        for (int k = lane; k < t; k += 32) th[k] = theta[pt * t + k];
        for (int k = lane; k < Wd; k += 32) wmask[k] = 0ull;
        __syncwarp();
        for (int r = lane; r < mi; r += 32) {
            const double* vr = P.V + (size_t)r * t1;
            double v = __ldg(vr);
            for (int k = 0; k < t; ++k) v = fma(__ldg(vr + 1 + k), th[k], v);
            w[r] = v;
            tolv[r] = PPG_QP_TOL * (1.0 + fabs(v));
        }
        __syncwarp();
        int nW = 0, j = -1, it = 0, status = -1;
        double lamj = 0.0;
        for (;;) {
            if (j < 0) {
                // most negative violated slack outside W, lowest row on ties
                double bv = INF;
                int best = 0x7fffffff;
                for (int r = lane; r < mi; r += 32) {
                    if ((wmask[r >> 6] >> (r & 63)) & 1ull) continue;
                    const double v = w[r];
                    if (v < -tolv[r] && v < bv) { bv = v; best = r; }
                }
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) {
                    const double ov = __shfl_xor_sync(0xffffffffu, bv, o);
                    const int oi = __shfl_xor_sync(0xffffffffu, best, o);
                    if (ov < bv || (ov == bv && oi < best)) { bv = ov; best = oi; }
                }
                best = __shfl_sync(0xffffffffu, best, 0);
                if (best == 0x7fffffff) { status = PPG_QP_OPTIMAL; break; }
                j = best;
                lamj = 0.0;
            }
            if (it >= PPG_QP_MAX_ITER) { status = PPG_QP_ITERLIM; break; }
            ++it;
            // forward solve L l = G_Wj (column-oriented: lanes update the rows below the pivot)
            for (int i = lane; i < nW; i += 32) g[i] = G[(size_t)widx[i] * mi + j];
            __syncwarp();
            for (int i = 0; i < nW; ++i) {
                const double gi = g[i] / L[k8_tri(i, i)];
                __syncwarp();
                if (lane == 0) g[i] = gi;
                for (int r = i + 1 + lane; r < nW; r += 32) g[r] = fma(-L[k8_tri(r, i)], gi, g[r]);
                __syncwarp();
            }
            double ll = 0.0;
            for (int i = lane; i < nW; i += 32) ll = fma(g[i], g[i], ll);
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) ll += __shfl_xor_sync(0xffffffffu, ll, o);
            ll = __shfl_sync(0xffffffffu, ll, 0);
            const double gjj = G[(size_t)j * mi + j], z = gjj - ll;
            // back solve L' d = -l
            for (int i = lane; i < nW; i += 32) d[i] = -g[i];
            __syncwarp();
            for (int i = nW - 1; i >= 0; --i) {
                const double di = d[i] / L[k8_tri(i, i)];
                __syncwarp();
                if (lane == 0) d[i] = di;
                for (int r = lane; r < i; r += 32) d[r] = fma(-L[k8_tri(i, r)], di, d[r]);
                __syncwarp();
            }
            const bool full = z > PPG_QP_CURV * gjj;
            const double sf = full ? -w[j] / z : INF;
            // ratio test over the multipliers of W, lowest row on ties
            double sb = INF;
            int brow = 0x7fffffff, bpos = -1;
            for (int i = lane; i < nW; i += 32) {
                const double di = d[i];
                if (!(di < -PPG_QP_DTOL)) continue;
                const double rt = lam[i] / -di;
                if (rt < sb || (rt == sb && widx[i] < brow)) { sb = rt; brow = widx[i]; bpos = i; }
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                const double ov = __shfl_xor_sync(0xffffffffu, sb, o);
                const int orow = __shfl_xor_sync(0xffffffffu, brow, o);
                const int opos = __shfl_xor_sync(0xffffffffu, bpos, o);
                if (ov < sb || (ov == sb && orow < brow)) { sb = ov; brow = orow; bpos = opos; }
            }
            sb = __shfl_sync(0xffffffffu, sb, 0);
            bpos = __shfl_sync(0xffffffffu, bpos, 0);
            if (bpos < 0 && !full) { status = PPG_QP_INFEASIBLE; break; }
            const bool partial = sb < sf;
            const double s = partial ? sb : sf;
            if (!isfinite(s)) { status = PPG_QP_NUMERIC; break; }
            // w += s (G[:,j] + G[:,W] d)
            for (int r = lane; r < mi; r += 32) {
                double u = G[(size_t)j * mi + r];
                for (int k = 0; k < nW; ++k) u = fma(G[(size_t)widx[k] * mi + r], d[k], u);
                w[r] = fma(s, u, w[r]);
            }
            for (int k = lane; k < nW; k += 32) lam[k] = fma(s, d[k], lam[k]);
            lamj += s;
            __syncwarp();
            if (partial) {
                const int p = bpos;
                for (int r = p + 1 + lane; r < nW; r += 32) xv[r - 1] = L[k8_tri(r, p)];
                __syncwarp();
                // rows below p move up one row without column p (row r - 1's new slot is exactly row r - 1's old one)
                for (int r = p + 1; r < nW; ++r) {
                    const int c0 = lane, c1 = lane + 32;
                    const double v0 = c0 <= r ? L[k8_tri(r, c0)] : 0.0, v1 = c1 <= r ? L[k8_tri(r, c1)] : 0.0;
                    __syncwarp();
                    if (c0 <= r && c0 != p) L[k8_tri(r - 1, c0 - (c0 > p))] = v0;
                    if (c1 <= r && c1 != p) L[k8_tri(r - 1, c1 - (c1 > p))] = v1;
                    __syncwarp();
                }
                // trailing block += x x'  (rank-one update, rows split over the lanes)
                bool ok = true;
                for (int k = p; k < nW - 1; ++k) {
                    const double lkk = L[k8_tri(k, k)], xk = xv[k];
                    const double rr = sqrt(fma(lkk, lkk, xk * xk)), c = rr / lkk, sn = xk / lkk;
                    __syncwarp();
                    for (int i = k + 1 + lane; i < nW - 1; i += 32) {
                        const double lik = (L[k8_tri(i, k)] + sn * xv[i]) / c;
                        L[k8_tri(i, k)] = lik;
                        xv[i] = c * xv[i] - sn * lik;
                    }
                    if (lane == 0) L[k8_tri(k, k)] = rr;
                    ok = ok && rr > 0.0 && isfinite(rr);
                    __syncwarp();
                }
                const int drop = widx[p];
                {
                    const int i0 = p + lane, i1 = p + 32 + lane;
                    const int a0 = i0 + 1 < nW ? widx[i0 + 1] : 0, a1 = i1 + 1 < nW ? widx[i1 + 1] : 0;
                    const double b0 = i0 + 1 < nW ? lam[i0 + 1] : 0.0, b1 = i1 + 1 < nW ? lam[i1 + 1] : 0.0;
                    __syncwarp();
                    if (i0 + 1 < nW) { widx[i0] = a0; lam[i0] = b0; }
                    if (i1 + 1 < nW) { widx[i1] = a1; lam[i1] = b1; }
                }
                if (lane == 0) wmask[drop >> 6] &= ~(1ull << (drop & 63));
                --nW;
                __syncwarp();
                if (!ok) { status = PPG_QP_NUMERIC; break; }
            } else {
                if (nW >= np) { status = PPG_QP_NUMERIC; break; }
                for (int i = lane; i < nW; i += 32) L[k8_tri(nW, i)] = g[i];
                if (lane == 0) {
                    L[k8_tri(nW, nW)] = sqrt(z);
                    widx[nW] = j;
                    lam[nW] = lamj;
                    wmask[j >> 6] |= 1ull << (j & 63);
                }
                ++nW;
                j = -1;
                __syncwarp();
            }
        }
        __syncwarp();
        if (lane == 0) status_out[pt] = (uint8_t)status;
        if (iters_out && lane == 0) iters_out[pt] = it;
        if (mask_out) for (int k = lane; k < Wd; k += 32) mask_out[pt * Wd + k] = wmask[k];
        if (!x_out && !dual_out) continue;
        if (status != PPG_QP_OPTIMAL) {
            if (x_out) for (int i = lane; i < n; i += 32) x_out[pt * n + i] = QNAN;
            if (dual_out) for (int i = lane; i < P.m; i += 32) dual_out[pt * P.m + i] = QNAN;
            continue;
        }
        for (int i = lane; i < n; i += 32) {
            const double* xr = P.Xp + (size_t)i * t1;
            double v = __ldg(xr);
            for (int k = 0; k < t; ++k) v = fma(__ldg(xr + 1 + k), th[k], v);
            for (int k = 0; k < nW; ++k) v = fma(-__ldg(P.K + (size_t)i * mi + widx[k]), lam[k], v);
            xo[i] = v;
            if (x_out) x_out[pt * n + i] = v;
        }
        if (!dual_out) continue;
        __syncwarp();
        for (int i = lane; i < n; i += 32) {
            double v = __ldg(P.c + i);
            for (int k = 0; k < t; ++k) v = fma(__ldg(P.H + (size_t)i * t + k), th[k], v);
            for (int k = 0; k < n; ++k) v = fma(__ldg(P.Q + (size_t)i * n + k), xo[k], v);
            for (int k = 0; k < nW; ++k) v = fma(__ldg(P.A + (size_t)(ne + widx[k]) * n + i), lam[k], v);
            ro[i] = v;
        }
        for (int r = lane; r < mi; r += 32) w[r] = 0.0;   // w is free now: the scattered lambda
        __syncwarp();
        for (int k = lane; k < nW; k += 32) w[widx[k]] = lam[k];
        for (int e = lane; e < ne; e += 32) {
            double v = 0.0;
            for (int i = 0; i < n; ++i) v = fma(__ldg(P.Pm + (size_t)e * n + i), ro[i], v);
            dual_out[pt * P.m + e] = -v;
        }
        __syncwarp();
        for (int r = lane; r < mi; r += 32) dual_out[pt * P.m + ne + r] = w[r];
    }
}

cudaError_t launch_theta_qp(const DevProgram& P, const double* theta, long long n_points, uint8_t* status, double* x,
                            double* dual, uint64_t* mask, int* iters, int sm_count, cudaStream_t st) {
    if (n_points <= 0) return cudaSuccess;
    if (!P.use_gram || P.np < 1 || P.np > 64) return cudaErrorInvalidValue;
    int dev = 0, lim = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&lim, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
    if (e != cudaSuccess) return e;
    const size_t warp_bytes = (size_t)k8_layout(P.mi, P.np, P.t, P.n, P.W).stride * sizeof(double);
    const size_t g_bytes = (((size_t)P.mi * P.mi + 1) & ~(size_t)1) * sizeof(double);
    const int stage_g = g_bytes + 4 * warp_bytes <= (size_t)lim;
    const size_t avail = (size_t)lim - (stage_g ? g_bytes : 0);
    int wpb = (int)(avail / warp_bytes);
    if (wpb > K8_MAX_WARPS) wpb = K8_MAX_WARPS;
    if (wpb < 1) return cudaErrorInvalidValue;
    const size_t smem = (stage_g ? g_bytes : 0) + (size_t)wpb * warp_bytes;
    if ((e = allow_max_smem(k8_theta_qp_kernel)) != cudaSuccess) return e;
    int per_sm = 0;
    if ((e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k8_theta_qp_kernel, wpb * 32, smem)) != cudaSuccess) return e;
    if (per_sm < 1) per_sm = 1;
    long long grid = (n_points + wpb - 1) / wpb;
    const long long cap = (long long)sm_count * per_sm;
    if (grid > cap) grid = cap;
    k8_theta_qp_kernel<<<(unsigned)grid, wpb * 32, smem, st>>>(P, theta, n_points, stage_g, status, x, dual, mask, iters);
    return cudaGetLastError();
}

}  // namespace ppgpu
