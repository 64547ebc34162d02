// K2a - feasibility CERTIFICATES by projected relaxation, one warp per candidate (runs before the K2 simplex).
//
// check_feasibility (/root/reference/src/ppopt/mplp_program.py:411-444) only asks whether
//   { z = (v, theta) : g_r z <= h_r  for all rows,  g_a z = h_a  for the active rows }
// is non-empty, and on every program of BASELINE.json 97-100 % of the candidates that survive the rank screen are
// feasible.  A feasible POINT is a complete proof, however it was found, so before paying for a simplex solve
// (K2: ~18 pivots x 112 x 38 fp64 FMAs in registers) every candidate gets a few dozen steps of the Agmon-Motzkin
// relaxation inside the affine subspace of its active rows:
//     i = most violated row,   z <- z - omega * (g_i z - h_i) / |N g_i|^2 * N g_i ,    N = projector onto null(G_A)
// All inner products come from the candidate-independent Gram matrix  Gam = G G'  (R0 x R0, built once per program):
//     residuals:  v <- v - tau * ( Gam[:,i] - Gam[:,A] w ),   w = (Gam[A,A])^-1 Gam[A,i]        (R0 x (1 + k') FMAs)
// i.e. ~8x less arithmetic per step than a simplex pivot, 40 registers per thread instead of 250, no block barrier.
// When the largest violation drops below PPG_FEAS_TOL the point is re-verified EXACTLY (every residual G z - h recomputed,
// equality residuals included) and only then is PPG_ST_FEAS set - the same acceptance rule as the LP (s* >= -1e-7).
// Candidates that do not converge within the step budget (all infeasible ones, and sets on which the projections
// zig-zag) are left for K2 - the register-resident kernel hands K2 the exact residuals of its last iterate, so the
// simplex starts from there (DevProgram::warm_*).  The relaxation never decides infeasibility.
// Two kernels: k2a_relax_reg_kernel (k' <= 8, R0 <= 128: the production path) and the generic k2a_relax_kernel.
#include "common.cuh"
#include "launch.h"
#include "lp_core.cuh"

#include <cstdlib>

namespace ppgpu {

__device__ __forceinline__ double dmax2(double a, double b) { return a > b ? a : b; }  // no NaN fix-up (fmax costs ~10 SASS)

constexpr double K2A_OMEGA = 1.35;  // scanned 1.2 .. 1.8 on the 100x30x6 program: fewest steps (32 vs 39 at 1.5)

template <int RPL>
__global__ void __launch_bounds__(128)
k2a_relax_kernel(DevProgram P, const uint64_t* __restrict__ masks, long long n, int k_act, uint8_t* __restrict__ status,
                 unsigned long long* __restrict__ queue, unsigned long long* __restrict__ counters, int max_iter) {
    extern __shared__ double dyn_smem[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int R0 = P.R0, nf = P.nfree, dc0 = P.dc0, W = P.W, k = k_act;
    // per-warp scratch: Sinv (k x k), ga (k), w (k), zs (nf), act (k ints)
    const size_t per_warp = (size_t)k * k + 2 * (size_t)k + (size_t)nf + (size_t)((k + 1) / 2 + 1);
    double* Sinv = dyn_smem + per_warp * warp;
    double* ga = Sinv + (size_t)k * k;
    double* wv = ga + k;
    double* zs = wv + k;
    int* act = reinterpret_cast<int*>(zs + nf);
    const double* __restrict__ Gam = P.Gam;
    const double* __restrict__ T0 = P.T0;
    unsigned long long n_try = 0, n_ok = 0, n_it = 0;
    for (;;) {
        unsigned long long q = 0;
        if (lane == 0) q = atomicAdd(queue, 1ull);
        const long long idx = (long long)__shfl_sync(PPG_FULL, q, 0);
        if (idx >= n) break;
        const uint8_t st = status[idx];
        if (!(st & PPG_ST_RANK) || (st & PPG_ST_FEAS)) continue;
        const uint64_t* mk = masks + idx * W;
        ++n_try;
        __syncwarp();
        for (int j = lane; j < k; j += 32) act[j] = mask_nth(mk, W, j);
        __syncwarp();
        // ---- S = Gam[A,A], Cholesky in place, then Sinv = S^-1 column by column
        for (int e = lane; e < k * k; e += 32) Sinv[e] = __ldg(Gam + (size_t)act[e / k] * R0 + act[e % k]);
        __syncwarp();
        bool pd = true;
        for (int j = 0; j < k; ++j) {
            const double d = Sinv[j * k + j];
            if (!(d > 1e-300)) { pd = false; break; }
            const double sd = sqrt(d);
            __syncwarp();
            for (int i = j + 1 + lane; i < k; i += 32) Sinv[i * k + j] /= sd;
            if (lane == 0) Sinv[j * k + j] = sd;
            __syncwarp();
            for (int i = j + 1 + lane; i < k; i += 32) {
                const double lij = Sinv[i * k + j];
                for (int c = j + 1; c <= i; ++c) Sinv[i * k + c] = fma(-lij, Sinv[c * k + j], Sinv[i * k + c]);
            }
            __syncwarp();
        }
        if (!pd) continue;
        {
            // lane c solves L L' x = e_c; the lower triangle holds L, results go to the upper part via registers
            double x[32];
            const int c = lane;
            if (c < k) {
#pragma unroll 1
                for (int i = 0; i < k; ++i) {
                    double s = (i == c) ? 1.0 : 0.0;
                    for (int j = 0; j < i; ++j) s = fma(-Sinv[i * k + j], x[j], s);
                    x[i] = s / Sinv[i * k + i];
                }
#pragma unroll 1
                for (int i = k - 1; i >= 0; --i) {
                    double s = x[i];
                    for (int j = i + 1; j < k; ++j) s = fma(-Sinv[j * k + i], x[j], s);
                    x[i] = s / Sinv[i * k + i];
                }
            }
            __syncwarp();
            if (c < k) for (int i = 0; i < k; ++i) Sinv[i * k + c] = x[i];
            __syncwarp();
        }
        // ---- start point: minimum-norm solution of the active equalities  z0 = G_A' Sinv h_A
        for (int a = lane; a < k; a += 32) ga[a] = __ldg(T0 + (size_t)act[a] * dc0);
        __syncwarp();
        for (int a = lane; a < k; a += 32) {
            double s = 0.0;
            for (int b = 0; b < k; ++b) s = fma(Sinv[a * k + b], ga[b], s);
            wv[a] = s;
        }
        __syncwarp();
        double z[2];
#pragma unroll
        for (int cc = 0; cc < 2; ++cc) {
            const int c = cc * 32 + lane;
            double s = 0.0;
            if (c < nf) for (int a = 0; a < k; ++a) s = fma(__ldg(T0 + (size_t)act[a] * dc0 + 1 + c), wv[a], s);
            z[cc] = s;
            if (c < nf) zs[c] = s;
        }
        __syncwarp();
        double v[RPL];
        bool isA[RPL];
        auto exact_residuals = [&]() {
#pragma unroll
            for (int rr = 0; rr < RPL; ++rr) {
                const int r = rr * 32 + lane;
                double s = 0.0;
                if (r < R0) {
                    const double* g = T0 + (size_t)r * dc0;
                    s = -__ldg(g);
                    for (int c = 0; c < nf; ++c) s = fma(__ldg(g + 1 + c), zs[c], s);
                }
                v[rr] = s;
            }
        };
#pragma unroll
        for (int rr = 0; rr < RPL; ++rr) {
            const int r = rr * 32 + lane;
            isA[rr] = r < P.mi && mask_test(mk, r);
        }
        exact_residuals();
        __syncwarp();  // zs is rewritten by the first re-verification
        bool feasible = false;
        int rechecks = 0;
        for (int it = 0; it < max_iter; ++it) {
            // most violated inequality row
            double lv = 0.0;
#pragma unroll
            for (int rr = 0; rr < RPL; ++rr)
                if (!isA[rr] && rr * 32 + lane < R0) lv = fmax(lv, v[rr]);
            const double wmax = warp_max_nonneg(lv);
            if (wmax <= PPG_FEAS_TOL) {
                // exact re-verification from the point itself (also checks the equality residuals)
#pragma unroll
                for (int cc = 0; cc < 2; ++cc) if (cc * 32 + lane < nf) zs[cc * 32 + lane] = z[cc];
                __syncwarp();
                exact_residuals();
                __syncwarp();  // zs is rewritten by a later re-verification
                double worst = 0.0;
#pragma unroll
                for (int rr = 0; rr < RPL; ++rr)
                    if (rr * 32 + lane < R0) worst = fmax(worst, isA[rr] ? fabs(v[rr]) : v[rr]);
                worst = warp_max_nonneg(fmax(worst, 0.0));
                if (worst <= PPG_FEAS_TOL) { feasible = true; break; }
                if (++rechecks > 3) break;
                continue;
            }
            int irow = 0x7fffffff;
#pragma unroll
            for (int rr = RPL - 1; rr >= 0; --rr) {
                const unsigned m = __ballot_sync(PPG_FULL, !isA[rr] && rr * 32 + lane < R0 && v[rr] == wmax);
                if (m) irow = rr * 32 + __ffs((int)m) - 1;
            }
            ++n_it;
            // w = Sinv * Gam[A, i]
            for (int a = lane; a < k; a += 32) ga[a] = __ldg(Gam + (size_t)act[a] * R0 + irow);
            __syncwarp();
            for (int a = lane; a < k; a += 32) {
                double s = 0.0;
                for (int b = 0; b < k; ++b) s = fma(Sinv[a * k + b], ga[b], s);
                wv[a] = s;
            }
            __syncwarp();
            double nn = __ldg(Gam + (size_t)irow * R0 + irow);
            const double gii = nn;
            for (int a = 0; a < k; ++a) nn = fma(-ga[a], wv[a], nn);
            if (!(nn > 1e-12 * gii)) break;  // row i is (numerically) in the span of the active rows: leave it to the LP
            const double tau = K2A_OMEGA * wmax / nn;
#pragma unroll
            for (int rr = 0; rr < RPL; ++rr) {
                const int r = rr * 32 + lane;
                if (r < R0) {
                    double col = __ldg(Gam + (size_t)irow * R0 + r);
                    for (int a = 0; a < k; ++a) col = fma(-__ldg(Gam + (size_t)act[a] * R0 + r), wv[a], col);
                    v[rr] = fma(-tau, col, v[rr]);
                }
            }
#pragma unroll
            for (int cc = 0; cc < 2; ++cc) {
                const int c = cc * 32 + lane;
                if (c < nf) {
                    double d = __ldg(T0 + (size_t)irow * dc0 + 1 + c);
                    for (int a = 0; a < k; ++a) d = fma(-__ldg(T0 + (size_t)act[a] * dc0 + 1 + c), wv[a], d);
                    z[cc] = fma(-tau, d, z[cc]);
                }
            }
            __syncwarp();  // ga / wv are rewritten by the next step
        }
        if (feasible) {
            ++n_ok;
            if (lane == 0) status[idx] = st | PPG_ST_FEAS;
        }
    }
    if (lane == 0 && n_try) {
        atomicAdd(&counters[CNT_K2A_TRIED], n_try);
        atomicAdd(&counters[CNT_K2A_CERTIFIED], n_ok);
        atomicAdd(&counters[CNT_K2A_STEPS], n_it);
        atomicAdd(&counters[CNT_K2A_WORK], n_it * (unsigned long long)(R0 * (k + 1)));
    }
}

template <int RPL>
static cudaError_t launch_k2a_t(const DevProgram& P, const uint64_t* masks, long long n, int k_act, uint8_t* status,
                                unsigned long long* queue, unsigned long long* counters, int max_iter, int sm_count,
                                cudaStream_t st) {
    auto kern = k2a_relax_kernel<RPL>;
    const size_t per_warp = (size_t)k_act * k_act + 2 * (size_t)k_act + (size_t)P.nfree + (size_t)((k_act + 1) / 2 + 1);
    const size_t smem = per_warp * 4 * sizeof(double);
    cudaError_t e;
    if ((e = fit_smem(kern, smem)) != cudaSuccess) return e;
    int occ = 0;
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, 128, smem);
    if (e != cudaSuccess) return e;
    if (occ < 1) occ = 1;
    long long grid = (long long)sm_count * occ;
    const long long need = (n + 3) / 4;
    if (grid > need) grid = need;
    if (grid < 1) grid = 1;
    kern<<<(unsigned)grid, 128, smem, st>>>(P, masks, n, k_act, status, queue, counters, max_iter);
    return cudaGetLastError();
}


// ---------------------------------------------------------------------------------------------------------------------
// Register-resident variant for small active sets (k' <= 8, R0 <= 128): everything candidate-specific lives in registers.
//   * Gam[A,A] is factorised as L D L' by every lane redundantly (k' <= 8: ~60 FMAs, no shared memory, no __syncwarp,
//     no sqrt and k' reciprocals instead of 3k' divisions), M's rows are triangular solves against it;
//   * the point is carried as the log of its steps (tau_e, row i_e): z = -sum_e tau_e g_{i_e} + G_A' x - one shared
//     memory store per step, no read;
//   * arg-max of the violations in ONE 32-bit reduction: key = high word of the violation with the row index in its 7
//     lowest bits (13 mantissa bits are plenty for a number that only steers the relaxation);
//   * the exact verification stays in Gram space: residual_r = sum_j c_j Gam[j,r] + sum_a x_a Gam[A_a,r] - h_r with
//     x = S^-1 (h_A - Gam[A,T] c_T) - coalesced row reads of Gam, every row recomputed (not only near-binding ones),
//     equality residuals included; same acceptance rule, rounding error ~1e-15 like the z-space evaluation.
// Rows r >= R0 of a lane are parked at -1e300 and read past the end of a Gam row (the program arrays carry a 1 KiB
// zero tail, api.cu upload()), which keeps the hot loop free of clamps and bounds predicates.
template <int KC>
__device__ __forceinline__ void ldl_solve(const double (&L)[KC][KC], const double (&dinv)[KC], double (&x)[KC]) {
#pragma unroll
    for (int i = 1; i < KC; ++i) {
#pragma unroll
        for (int c = 0; c < KC; ++c) if (c < i) x[i] = fma(-L[i][c], x[c], x[i]);
    }
#pragma unroll
    for (int i = 0; i < KC; ++i) x[i] *= dinv[i];
#pragma unroll
    for (int i = KC - 2; i >= 0; --i) {
#pragma unroll
        for (int c = 0; c < KC; ++c) if (c > i) x[i] = fma(-L[c][i], x[c], x[i]);
    }
}

__device__ __forceinline__ double k2a_key(double v, int idx) {
    return __hiloint2double(__double2hiint(v), (__double2loint(v) & ~127) | idx);
}

constexpr int K2A_LOG = 192;       // step log entries per warp (both phases together are clamped to it)
constexpr double K2A_OMEGA2 = 1.8; // second phase, see the step loop
constexpr int K2A_STALL2 = 48;

template <int RPL, int KC, bool EXACT>
__global__ void __launch_bounds__(128, (RPL * KC <= 16) ? 5 : ((RPL * KC <= 24) ? 4 : 3))   // 96 registers for 4 x 5 spill M: slower
k2a_relax_reg_kernel(DevProgram P, const uint64_t* __restrict__ masks, long long n, int k_act, uint8_t* __restrict__ status,
                     unsigned long long* __restrict__ queue, unsigned long long* __restrict__ counters, int max_iter, int max_iter2,
                     int grab) {
    constexpr int NL = KC * (KC - 1) / 2;
    __shared__ double fac_s[4][NL + KC];   // per warp: strict lower triangle of L (row-major), then 1/d
    __shared__ double log_s[4][K2A_LOG];   // per warp: tau of every step, stepped row in the 7 low mantissa bits
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int R0 = P.R0, dc0 = P.dc0, W = P.W, k = EXACT ? KC : k_act;
    double* fac = fac_s[warp];
    double* lg = log_s[warp];
    unsigned lg_sa = (unsigned)__cvta_generic_to_shared(lg);
    asm volatile("" : "+r"(lg_sa));
    const double* __restrict__ Gam = P.Gam;
    const double* __restrict__ T0 = P.T0;
    if (max_iter > K2A_LOG) max_iter = K2A_LOG;
    if (max_iter + max_iter2 > K2A_LOG) max_iter2 = K2A_LOG - max_iter;
    // a key <= ktol proves violation < PPG_FEAS_TOL (keys round down by < 2^-13 relative): time for the exact verification
    const int ktol = (__double2hiint(PPG_FEAS_TOL * 0.999) & ~127) | 127;
    // opaque per-lane constants (kept in registers instead of being rematerialised inside the step loop)
    unsigned long long glane = (unsigned long long)(Gam + lane);
    asm volatile("" : "+l"(glane));
    int kid[RPL];
#pragma unroll
    for (int rr = 0; rr < RPL; ++rr) { kid[rr] = rr * 32 + lane; asm volatile("" : "+r"(kid[rr])); }
    unsigned long long n_try = 0, n_ok = 0, n_it = 0;
    // A warp takes `grab` (<= 32) consecutive candidates per queue item: lanes fetch the status byte and the mask words of one
    // of them each up front (the two dependent HBM round trips and the atomic are paid once per item, not per candidate),
    // the masks wait in shared memory, and the candidates that need work are then processed one after the other.
    // The host picks grab = 32 for large launches and less for small ones, so that every warp still sees >= 16 items.
    __shared__ uint64_t mk_s[4][32 * 4];
    for (;;) {
        unsigned long long q = 0;
        if (lane == 0) q = atomicAdd(queue, (unsigned long long)grab);
        const long long base = (long long)__shfl_sync(PPG_FULL, q, 0);
        if (base >= n) break;
        uint8_t st_l = 0;
        __syncwarp();   // the previous batch's masks are no longer read
        if (lane < grab && base + lane < n) {
            st_l = status[base + lane];
            for (int w = 0; w < W; ++w) mk_s[warp][lane * 4 + w] = masks[(base + lane) * W + w];
        }
        __syncwarp();
        unsigned todo = __ballot_sync(PPG_FULL, (st_l & PPG_ST_RANK) && !(st_l & PPG_ST_FEAS));
        while (todo) {
        const int bj = __ffs((int)todo) - 1;
        todo &= todo - 1;
        const long long idx = base + bj;
        const uint8_t st = (uint8_t)__shfl_sync(PPG_FULL, (int)st_l, bj);
        const uint64_t* mk = &mk_s[warp][bj * 4];
        ++n_try;
        // ---- active rows: lane a < k finds the a-th set bit, everybody gets all of them (padded slots repeat row 0)
        const int act_lane = mask_nth(mk, W, lane < k ? lane : 0);
        int act[KC];
        unsigned gp[KC];   // element offset of Gam[act[a], 0] (32 bits: half the registers of a pointer)
#pragma unroll
        for (int a = 0; a < KC; ++a) {
            act[a] = __shfl_sync(PPG_FULL, act_lane, (EXACT || a < k) ? a : 0);
            gp[a] = (unsigned)act[a] * (unsigned)R0;
            asm volatile("" : "+r"(gp[a]));
        }
#define K2A_GP(a, off) __ldg(Gam + (gp[a] + (unsigned)(off)))
        // ---- S = Gam[A,A] = L D L' (unit lower L), computed redundantly by every lane; padded slots form an identity block
        double L[KC][KC], dinv[KC];
        bool pd = true;
        {
            double dd[KC];
#pragma unroll
            for (int i = 0; i < KC; ++i) {
#pragma unroll
                for (int j = 0; j < KC; ++j) {
                    if (j <= i) {
                        const double e = (EXACT || (i < k && j < k)) ? K2A_GP(i, act[j]) : (i == j ? 1.0 : 0.0);
                        if (j == i) dd[i] = e; else L[i][j] = e;
                    }
                }
            }
#pragma unroll
            for (int j = 0; j < KC; ++j) {
                double wj[KC];
#pragma unroll
                for (int c = 0; c < KC; ++c) if (c < j) { wj[c] = L[j][c] * dd[c]; dd[j] = fma(-L[j][c], wj[c], dd[j]); }
                pd = pd && (dd[j] > 1e-300);
                dinv[j] = 1.0 / dd[j];
#pragma unroll
                for (int i = 0; i < KC; ++i) {
                    if (i > j) {
                        double e = L[i][j];
#pragma unroll
                        for (int c = 0; c < KC; ++c) if (c < j) e = fma(-L[i][c], wj[c], e);
                        L[i][j] = e * dinv[j];
                    }
                }
            }
        }
        if (!pd) continue;  // uniform: every lane computed the same factorisation
        __syncwarp();       // the previous candidate's verification may still be reading fac
        if (lane == 0) {
            int o = 0;
#pragma unroll
            for (int i = 0; i < KC; ++i) {
#pragma unroll
                for (int j = 0; j < KC; ++j) if (j < i) fac[o++] = L[i][j];
            }
#pragma unroll
            for (int i = 0; i < KC; ++i) fac[NL + i] = dinv[i];
        }
        // ---- start point: min-norm solution of the active equalities, z0 = G_A' w0
        double w0[KC];
#pragma unroll
        for (int a = 0; a < KC; ++a) w0[a] = (EXACT || a < k) ? __ldg(T0 + (size_t)act[a] * dc0) : 0.0;
        ldl_solve<KC>(L, dinv, w0);
        // ---- per-lane rows: M = Gam[:,A] S^-1 and the start residuals
        double M[RPL][KC], v[RPL];
        unsigned amask = 0;  // bit rr: row rr*32+lane is one of the active rows
#pragma unroll
        for (int rr = 0; rr < RPL; ++rr) {
            const int r = rr * 32 + lane;
            double x[KC];
#pragma unroll
            for (int a = 0; a < KC; ++a) x[a] = (EXACT || a < k) ? K2A_GP(a, r) : 0.0;
            double s2 = -__ldg(T0 + (size_t)min(r, R0 - 1) * dc0);
#pragma unroll
            for (int a = 0; a < KC; ++a) s2 = fma(x[a], w0[a], s2);
            ldl_solve<KC>(L, dinv, x);
#pragma unroll
            for (int a = 0; a < KC; ++a) M[rr][a] = x[a];
            const bool isa = r < P.mi && mask_test(mk, r);
            amask |= (isa ? 1u : 0u) << rr;
            v[rr] = (r < R0 && !isa) ? s2 : -1e300;  // parked: never the maximum
        }
        bool feasible = false;
        int rechecks = 0, nlog = 0, wref = 0;
        // exact residuals of the current iterate in Gram space (see header of this kernel): replay the step log
        auto exact_residuals = [&](double (&s)[RPL]) {
            __syncwarp();   // lane 0's fac stores, everybody's log stores
#pragma unroll
            for (int rr = 0; rr < RPL; ++rr) s[rr] = -__ldg(T0 + (size_t)min(rr * 32 + lane, R0 - 1) * dc0);
            double t = 0.0;  // lanes < k: Gam[A_lane, T] c_T
            const unsigned long long gact = (unsigned long long)(Gam + act_lane);
            for (int e = 0; e < nlog; ++e) {
                const double tk = lg[e];
                const unsigned off = (unsigned)((__double2loint(tk) & 127) * R0);
                const double* rp = reinterpret_cast<const double*>(glane) + off;
#pragma unroll
                for (int r2 = 0; r2 < RPL; ++r2) s[r2] = fma(-tk, __ldg(rp + r2 * 32), s[r2]);
                t = fma(-tk, __ldg(reinterpret_cast<const double*>(gact) + off), t);
            }
            const double rb = __ldg(T0 + (size_t)act_lane * dc0) - t;
            double x[KC];
#pragma unroll
            for (int b = 0; b < KC; ++b) {
                x[b] = shfl_d(rb, b);
                if (!EXACT && b >= k) x[b] = 0.0;
            }
            {
                double Lv[KC][KC], dv[KC];
                int o = 0;
#pragma unroll
                for (int i = 0; i < KC; ++i) {
#pragma unroll
                    for (int j = 0; j < KC; ++j) if (j < i) Lv[i][j] = fac[o++];
                }
#pragma unroll
                for (int i = 0; i < KC; ++i) dv[i] = fac[NL + i];
                ldl_solve<KC>(Lv, dv, x);
            }
#pragma unroll
            for (int a = 0; a < KC; ++a) {
#pragma unroll
                for (int r2 = 0; r2 < RPL; ++r2) s[r2] = fma(x[a], K2A_GP(a, lane + r2 * 32), s[r2]);
            }
        };
        // Two phases.  omega = 1.35 minimises the steps of the candidates that converge (scanned 1.2 .. 1.8); the ones that
        // stall with it (not halving the worst violation in 16 steps: fat sets on which the projections zig-zag) mostly
        // do converge with a longer stride, so a stall - or the end of the first budget - switches to omega = 1.8 for up to
        // max_iter2 more steps before the candidate is handed to the simplex (emulated on the CPU first: 4.9 % -> 1.5 %
        // uncertified for 7 % more steps; omega = 1.8 from the start costs 20 % more steps on everything).
        double omega = K2A_OMEGA;
        int it_end = max_iter, chk = 0;
        bool second = max_iter2 <= 0;   // "already in the last phase"
        for (int it = 0;; ++it) {
            // arg-max in one 32-bit reduction: the key of a residual is the high word of the double with the row index in
            // its 7 low bits (parked and satisfied rows have negative keys)
            int kmax = 0;
#pragma unroll
            for (int rr = 0; rr < RPL; ++rr) kmax = max(kmax, (__double2hiint(v[rr]) & ~127) | kid[rr]);
            const int wkey = __reduce_max_sync(PPG_FULL, kmax);
            if (wkey <= ktol) {
                // ---- exact verification
                double s[RPL];
                exact_residuals(s);
                double worst = 0.0;
#pragma unroll
                for (int rr = 0; rr < RPL; ++rr) {
                    const int r = rr * 32 + lane;
                    const bool isa = (amask >> rr) & 1u;
                    if (r < R0) worst = dmax2(worst, isa ? fabs(s[rr]) : s[rr]);
                    v[rr] = (r < R0 && !isa) ? s[rr] : -1e300;
                }
                worst = warp_max_nonneg(dmax2(worst, 0.0));
                if (worst <= PPG_FEAS_TOL) { feasible = true; break; }
                if (++rechecks > 3) break;
                continue;
            }
            const int irow = wkey & 127;   // a most violated row (to 13 mantissa bits)
            const int wl = irow & 31, wslot = irow >> 5;
            const double wmax = __hiloint2double(wkey & ~127, 0);   // its violation, rounded down by < 2^-13
            // stall detector: a relaxation that has not halved its worst violation in 16 steps is not going to finish
            // inside the budget (badly scaled or zero-margin sets) -> simplex.  Halving = exponent - 1 = key - 2^20.
            bool stalled = it >= it_end;
            if (!stalled && chk == 0) {
                stalled = it != 0 && wkey > wref - 0x100000;
                wref = wkey;
                chk = second ? K2A_STALL2 : 16;
            }
            if (stalled) {
                if (second) break;
                second = true;
                omega = K2A_OMEGA2;
                it_end = it + max_iter2;
                wref = wkey;
                chk = K2A_STALL2;
            }
            --chk;
            double g2[KC];
#pragma unroll
            for (int a = 0; a < KC; ++a) g2[a] = K2A_GP(a, irow);  // broadcast loads (padded slots: M == 0)
            const double* rowp = reinterpret_cast<const double*>(glane) + (unsigned)(irow * R0);
            double c2[RPL];
#pragma unroll
            for (int rr = 0; rr < RPL; ++rr) {
                double x2 = __ldg(rowp + rr * 32);
#pragma unroll
                for (int a = 0; a < KC; ++a) x2 = fma(-M[rr][a], g2[a], x2);
                c2[rr] = x2;
            }
            double mycol = c2[0];
#pragma unroll
            for (int rr = 1; rr < RPL; ++rr) if (rr == wslot) mycol = c2[rr];
            const double nn = shfl_d(mycol, wl);   // |N g_i|^2
            if (!(nn > 1e-12)) break;              // row i lies in the span of the active rows: leave it to the LP
            // z -= tau (g_i - G_A' w).  tau needs no accuracy; its low mantissa bits carry the row
            double rnn;   // gross (20-bit) reciprocal: one MUFU instead of convert - rcp - convert
            asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(rnn) : "d"(nn));
            const double tau = k2a_key((omega * wmax) * rnn, irow);
            // predicated store by lane 0 (no branch; every lane holds the same tau)
            asm volatile("{ .reg .pred p; setp.eq.s32 p, %2, 0; @p st.shared.f64 [%0], %1; }"
                         :: "r"(lg_sa + 8u * (unsigned)nlog), "d"(tau), "r"(lane) : "memory");
            ++nlog;
#pragma unroll
            for (int rr = 0; rr < RPL; ++rr) v[rr] = fma(-tau, c2[rr], v[rr]);
        }
        n_it += (unsigned)nlog;
        if (feasible) {
            ++n_ok;
            if (lane == 0) status[idx] = st | PPG_ST_FEAS;
        } else if (P.warm_count != nullptr) {
            // not certified: hand the last iterate to the simplex as its origin (exact residuals, any point will do)
            double s[RPL];
            exact_residuals(s);
            unsigned long long slot = 0;
            if (lane == 0) slot = atomicAdd(P.warm_count, 1ull);
            slot = __shfl_sync(PPG_FULL, slot, 0);
            bool fin = true;
#pragma unroll
            for (int rr = 0; rr < RPL; ++rr) fin = fin && (rr * 32 + lane >= R0 || fabs(s[rr]) < 1e300);
            fin = __all_sync(PPG_FULL, fin);
            if (slot < (unsigned long long)P.warm_cap) {   // every slot handed out below the cap gets an index (-1: unused)
#pragma unroll
                for (int rr = 0; rr < RPL; ++rr)
                    if (fin && rr * 32 + lane < R0) P.warm_resid[slot * (unsigned long long)R0 + rr * 32 + lane] = s[rr];
                if (lane == 0) {
                    P.warm_idx[slot] = fin ? idx : -1;
                    if (fin) status[idx] = st | PPG_ST_PRE;
                }
            }
        }
#undef K2A_GP
        }
    }
    if (lane == 0 && n_try) {
        atomicAdd(&counters[CNT_K2A_TRIED], n_try);
        atomicAdd(&counters[CNT_K2A_CERTIFIED], n_ok);
        atomicAdd(&counters[CNT_K2A_STEPS], n_it);
        atomicAdd(&counters[CNT_K2A_WORK], n_it * (unsigned long long)(R0 * (k + 1)));
    }
}

template <int RPL, int KC, bool EXACT>
static cudaError_t launch_k2a_reg(const DevProgram& P, const uint64_t* masks, long long n, int k_act, uint8_t* status,
                                  unsigned long long* queue, unsigned long long* counters, int max_iter, int sm_count,
                                  cudaStream_t st) {
    auto kern = k2a_relax_reg_kernel<RPL, KC, EXACT>;
    int occ = 0;
    cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, 128, 0);
    if (e != cudaSuccess) return e;
    if (occ < 1) occ = 1;
    long long grid = (long long)sm_count * occ;
    // candidates per warp and queue item: 32 when every warp still gets >= 16 items, fewer for small launches (a warp that
    // draws one item more than its neighbours is the tail of the launch)
    int grab = 32;
    while (grab > 2 && n / grab < 16 * grid * 4) grab >>= 1;
    const long long need = (n + 4ll * grab - 1) / (4ll * grab);
    if (grid > need) grid = need;
    if (grid < 1) grid = 1;
    static const int iters2 = getenv("PPGPU_K2A_ITERS2") ? atoi(getenv("PPGPU_K2A_ITERS2")) : 96;
    kern<<<(unsigned)grid, 128, 0, st>>>(P, masks, n, k_act, status, queue, counters, max_iter, iters2, grab);
    return cudaGetLastError();
}

template <int KC>
static cudaError_t launch_k2a_reg_k(const DevProgram& P, const uint64_t* masks, long long n, int k_act, uint8_t* status,
                                    unsigned long long* queue, unsigned long long* counters, int max_iter, int sm_count,
                                    cudaStream_t st) {
#define K2A_REG(RPLV)                                                                                                       \
    return k_act == KC ? launch_k2a_reg<RPLV, KC, true>(P, masks, n, k_act, status, queue, counters, max_iter, sm_count, st) \
                       : launch_k2a_reg<RPLV, KC, false>(P, masks, n, k_act, status, queue, counters, max_iter, sm_count, st);
    if (P.R0 <= 32) { K2A_REG(1) }
    if (P.R0 <= 64) { K2A_REG(2) }
    K2A_REG(4)
#undef K2A_REG
}

cudaError_t launch_k2a(const DevProgram& P, const uint64_t* masks, long long n, int k_act, uint8_t* status,
                       unsigned long long* queue, unsigned long long* counters, int max_iter, int sm_count, cudaStream_t st) {
    if (k_act > 32 || P.nfree > 64) return cudaSuccess;  // outside the certificate kernel's envelope: K2 decides alone
    {
        // production path: Gram matrix projected once per prefix in shared memory, half a warp per candidate (k2p_prefix.cu)
        bool handled = false;
        const cudaError_t e = launch_k2a_prefix(P, masks, n, k_act, status, queue, counters, max_iter, sm_count, st, &handled);
        if (e != cudaSuccess || handled) return e;
    }
    if (k_act >= 1 && k_act <= 8 && P.R0 <= 128) {
        if (k_act <= 3) return launch_k2a_reg_k<3>(P, masks, n, k_act, status, queue, counters, max_iter, sm_count, st);
        if (k_act == 4) return launch_k2a_reg_k<4>(P, masks, n, k_act, status, queue, counters, max_iter, sm_count, st);
        if (k_act == 5) return launch_k2a_reg_k<5>(P, masks, n, k_act, status, queue, counters, max_iter, sm_count, st);
        if (k_act == 6) return launch_k2a_reg_k<6>(P, masks, n, k_act, status, queue, counters, max_iter, sm_count, st);
        return launch_k2a_reg_k<8>(P, masks, n, k_act, status, queue, counters, max_iter, sm_count, st);
    }
    if (P.R0 <= 32) return launch_k2a_t<1>(P, masks, n, k_act, status, queue, counters, max_iter, sm_count, st);
    if (P.R0 <= 64) return launch_k2a_t<2>(P, masks, n, k_act, status, queue, counters, max_iter, sm_count, st);
    if (P.R0 <= 128) return launch_k2a_t<4>(P, masks, n, k_act, status, queue, counters, max_iter, sm_count, st);
    if (P.R0 <= 256) return launch_k2a_t<8>(P, masks, n, k_act, status, queue, counters, max_iter, sm_count, st);
    return cudaSuccess;
}

}  // namespace ppgpu
