// K3 + K4, compact form - the same screen as k34_kkt.cu::k34_kernel (KKT by Schur complement, theta-space polytope,
// Chebyshev LP; reference: check_optimality /root/reference/src/ppopt/mpqp_program.py:203-322, region rows + filters
// utils/mpqp_utils.py:111-126, is_full_dimensional utils/mpqp_utils.py:323-344 -> utils/chebyshev_ball.py:10-63), written
// for the INSTRUCTION CACHE instead of for registers.
//
// k34_kernel keeps the R0 x (t+2) tableau in registers and pays for it with 6.7 k SASS instructions of fully unrolled
// row/column code (107 KB): with four warps per CTA at unrelated program counters the kernel is instruction-fetch bound
// (ncu r01/r02: stall_no_instruction 6.0 per issued instruction, issue slots 23 % busy, ~320 k cycles per candidate for
// ~10 k cycles of arithmetic).  Here the tableau of a candidate lives in SHARED memory (R0 x (t+2) doubles = 7 KB at the
// 100 x 30 x 6 program, odd row stride -> lanes over rows are bank-conflict free), every loop over rows / columns is a real
// loop, and the whole kernel is a few hundred instructions that stay in the L0/L1 instruction caches.
//
// The LP is the same LP with the same pivoting rules as lp_core.cuh (first pivot: r enters on the row of smallest right-
// hand side; then Dantzig pricing over free / slack columns, Harris ratio test with the largest pivot inside the band,
// Bland after PPG_BLAND_AFTER degenerate steps, rows whose basic variable is free are dropped, early exit as soon as the
// radius reaches the threshold) in plain dictionary form
//      w_i = b_i - sum_c A_ic x_c   (live rows),      maximise  z = beta - sum_c alpha_c x_c.
#include "common.cuh"
#include "launch.h"
#include "lp_core.cuh"

#include <algorithm>
#include <cstdlib>

namespace ppgpu {

struct K4cOut { int code; double beta; int pivots; long long work; };

// Chebyshev LP of one candidate on the warp's shared-memory tableau.  Tab: m x lds, column 0 = rhs, 1..t = theta, t+1 = r.
// flag[i]: 1 live row (basic slack), 0 dead.  Uniform result.
// 1 / x to full double precision without the IEEE division sequence (x: a pivot / ratio denominator, normal and non-zero)
__device__ __forceinline__ double k4c_rcp(double x) {
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
    r = r * fma(-x, r, 2.0);
    return r * fma(-x, r, 2.0);
}

__device__ __noinline__ K4cOut k4c_solve(double* __restrict__ Tab, unsigned char* __restrict__ flag, int* __restrict__ bvar,
                                         double* __restrict__ alpha, int* __restrict__ kind, int* __restrict__ nbv,
                                         double* __restrict__ prow, int m, int t, int lds, double thr, int lane) {
    const int nc = t + 1;            // nonbasic columns 1..nc (the last one is r)
    const int ld = nc + 1;
    K4cOut out; out.code = PPG_LP_OPTIMAL; out.beta = -CUDART_INF; out.pivots = 0; out.work = 0;
    int live = 0;
    #pragma unroll 1
    for (int i = lane; i < m; i += 32) { bvar[i] = ld + i; live += flag[i] ? 1 : 0; }
    live = __reduce_add_sync(PPG_FULL, live);
    #pragma unroll 1
    for (int c = lane; c < ld; c += 32) { alpha[c] = 0.0; kind[c] = (c >= 1) ? 1 : 0; nbv[c] = c; }   // kind: 1 free, 2 slack
    __syncwarp();
    double beta = 0.0;
    int degen = 0; bool bland = false;
    const int cap = 50 * (m + nc) + 200;
    for (int it = 0;; ++it) {
        int j, l; double dir = 1.0;
        if (it == 0) {
            // r enters on the row of smallest right-hand side (whatever its sign): afterwards every slack is >= 0
            double mn = CUDART_INF; int r0 = 0x7fffffff;
            #pragma unroll 1
            for (int i = lane; i < m; i += 32)
                if (flag[i]) { const double v = Tab[(size_t)i * lds]; if (v < mn) { mn = v; r0 = i; } }
            warp_argmin(mn, r0);
            if (r0 == 0x7fffffff) { out.code = PPG_LP_UNBOUNDED; out.beta = CUDART_INF; return out; }
            j = nc; l = r0;
            if (lane == 0) alpha[nc] = -1.0;   // z = r
            __syncwarp();
        } else {
            out.beta = beta;
            if (beta >= thr) { out.code = PPG_LP_EARLY; return out; }
            if (it > cap) { out.code = PPG_LP_ITERLIM; return out; }
            // ---- pricing (lanes over columns)
            double sc = 0.0; int key = 0x7fffffff, jc = 0x7fffffff;
            #pragma unroll 1
            for (int c = 1 + lane; c < ld; c += 32) {
                const double a = alpha[c];
                const double s2 = kind[c] == 1 ? fabs(a) : (kind[c] == 2 ? -a : 0.0);
                if (s2 > PPG_OPT_TOL) {
                    if (!bland) { if (s2 > sc) { sc = s2; jc = c; } }
                    else if (nbv[c] < key) { key = nbv[c]; jc = c; sc = s2; }
                }
            }
            if (!__any_sync(PPG_FULL, jc != 0x7fffffff)) { out.code = PPG_LP_OPTIMAL; return out; }
            if (!bland) {
                const double ws = warp_max_nonneg(sc);
                j = __reduce_min_sync(PPG_FULL, (jc != 0x7fffffff && sc == ws) ? jc : 0x7fffffff);
            } else {
                const int wk = __reduce_min_sync(PPG_FULL, key);
                j = __reduce_min_sync(PPG_FULL, key == wk ? jc : 0x7fffffff);
            }
            const double aj = alpha[j];
            const bool entering_free = kind[j] == 1;
            dir = (entering_free && aj > 0.0) ? -1.0 : 1.0;
            // ---- Harris ratio test (lanes over rows)
            double hb = CUDART_INF;
            #pragma unroll 1
            for (int i = lane; i < m; i += 32) {
                if (!flag[i]) continue;
                const double cv = dir * Tab[(size_t)i * lds + j];
                if (cv > PPG_TINY) {
                    const double rhs = fmax(Tab[(size_t)i * lds], 0.0);
                    hb = fmin(hb, (rhs + PPG_HARRIS) * k4c_rcp(cv));
                }
            }
            hb = warp_min_nonneg(hb);
            if (hb == CUDART_INF) { out.code = PPG_LP_UNBOUNDED; out.beta = CUDART_INF; return out; }
            double lp = 0.0, lr = CUDART_INF; int lrow = 0x7fffffff, lb = 0x7fffffff;
            #pragma unroll 1
            for (int i = lane; i < m; i += 32) {
                if (!flag[i]) continue;
                const double cv = dir * Tab[(size_t)i * lds + j];
                if (cv > PPG_TINY) {
                    const double rat = fmax(Tab[(size_t)i * lds], 0.0) * k4c_rcp(cv);
                    if (rat <= hb) {
                        const bool better = bland ? (bvar[i] < lb) : (cv > lp);
                        if (better) { lp = cv; lrow = i; lb = bvar[i]; lr = rat; }
                    }
                }
            }
            if (bland) {
                const int wb = __reduce_min_sync(PPG_FULL, lb);
                l = __reduce_min_sync(PPG_FULL, lb == wb ? lrow : 0x7fffffff);
            } else {
                const double wp = warp_max_nonneg(lp);
                l = __reduce_min_sync(PPG_FULL, (lrow != 0x7fffffff && lp == wp) ? lrow : 0x7fffffff);
            }
            if (l == 0x7fffffff) { out.code = PPG_LP_UNBOUNDED; out.beta = CUDART_INF; return out; }
            const double gr = __shfl_sync(PPG_FULL, lr, l & 31);
            if (gr <= PPG_DEGEN_STEP) { if (++degen > PPG_BLAND_AFTER) bland = true; } else degen = 0;
        }
        // ---- Gauss-Jordan exchange (row l, column j)
        const bool entering_free = kind[j] == 1;
        double* Tl = Tab + (size_t)l * lds;
        const double inv = k4c_rcp(Tl[j]);
        __syncwarp();
        #pragma unroll 1
        for (int c = lane; c < ld; c += 32) prow[c] = (c == j) ? 0.0 : Tl[c] * inv;
        __syncwarp();
        const double aj = alpha[j];
        #pragma unroll 1
        for (int i = lane; i < m; i += 32) {
            if (!flag[i] || i == l) continue;
            double* Ti = Tab + (size_t)i * lds;
            const double col = Ti[j];
            if (col != 0.0) {
                #pragma unroll 1
                for (int c = 0; c < ld; ++c) Ti[c] = fma(-col, prow[c], Ti[c]);
                Ti[j] = -col * inv;
            }
            if (Ti[0] < 0.0 && Ti[0] > -1e-9) Ti[0] = 0.0;
        }
        __syncwarp();
        beta = fma(-aj, prow[0], beta);
        #pragma unroll 1
        for (int c = 1 + lane; c < ld; c += 32) alpha[c] = (c == j) ? -aj * inv : fma(-aj, prow[c], alpha[c]);
        #pragma unroll 1
        for (int c = lane; c < ld; c += 32) Tl[c] = (c == j) ? inv : prow[c];
        out.pivots++; out.work += (long long)live * (nc + 1);
        if (lane == 0) {
            const int leave_var = bvar[l], enter_var = nbv[j];
            kind[j] = 2; nbv[j] = leave_var;
            if (entering_free) flag[l] = 0; else bvar[l] = enter_var;
        }
        if (entering_free) live--;
        __syncwarp();
    }
}

__global__ void __launch_bounds__(128)
k34c_kernel(DevProgram P, const uint64_t* __restrict__ masks, long long n, int k_act, uint8_t* __restrict__ status,
            unsigned long long* __restrict__ queue, unsigned long long* __restrict__ counters, int use_pre, int warp_bytes,
            int lds, int per_item) {
    extern __shared__ unsigned char k34c_smem[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int t = P.t, t1 = P.t + 1, mi = P.mi, W = P.W, k = k_act, m = P.R0;
    unsigned char* base = k34c_smem + (size_t)warp * warp_bytes;
    double* Tab = reinterpret_cast<double*>(base); base += (size_t)m * lds * 8;
    double* S = reinterpret_cast<double*>(base); base += (size_t)k * k * 8;
    double* Lam = reinterpret_cast<double*>(base); base += (size_t)k * t1 * 8;
    double* alpha = reinterpret_cast<double*>(base); base += (size_t)lds * 8;
    double* prow = reinterpret_cast<double*>(base); base += (size_t)lds * 8;
    int* act = reinterpret_cast<int*>(base); base += (size_t)((k + 1) & ~1) * 4;
    int* bvar = reinterpret_cast<int*>(base); base += (size_t)((m + 1) & ~1) * 4;
    int* kind = reinterpret_cast<int*>(base); base += (size_t)((lds + 1) & ~1) * 4;
    int* nbv = reinterpret_cast<int*>(base); base += (size_t)((lds + 1) & ~1) * 4;
    unsigned char* flag = base;
    unsigned long long n_lp = 0, n_piv = 0, n_work = 0, n_num = 0;
    const long long nblocks = (n + per_item - 1) / per_item;
    for (;;) {
        unsigned long long v = 0;
        if (lane == 0) v = atomicAdd(queue, 1ull);
        const long long item = (long long)__shfl_sync(PPG_FULL, v, 0);
        if (item >= nblocks) break;
        const long long c0 = item * per_item + lane;
        const uint8_t sb = (lane < per_item && c0 < n) ? status[c0] : 0;
        unsigned todo = __ballot_sync(PPG_FULL, (sb & PPG_ST_FEAS) && (!use_pre || (sb & PPG_ST_PRE)));
        while (todo) {
            const int src = __ffs((int)todo) - 1;
            todo &= todo - 1u;
            const long long idx = item * per_item + src;
            uint8_t st = (uint8_t)__shfl_sync(PPG_FULL, (int)sb, src);
            if (use_pre) st &= (uint8_t)~PPG_ST_PRE;
            const uint64_t* mk = masks + idx * W;
            __syncwarp();
            #pragma unroll 1
            for (int j = lane; j < k; j += 32) act[j] = mask_nth(mk, W, j);
            __syncwarp();
            #pragma unroll 1
            for (int e = lane; e < k * k; e += 32) {
                const int a = e / k, b2 = e - a * k;
                S[e] = __ldg(P.G + (size_t)act[a] * mi + act[b2]);
            }
            __syncwarp();
            // Cholesky (lower), right-looking, lanes over rows
            bool pd = true;
            #pragma unroll 1
            for (int j = 0; j < k; ++j) {
                const double d = S[j * k + j];
                if (!(d > 0.0)) { pd = false; break; }
                const double sd = sqrt(d);
                __syncwarp();
                #pragma unroll 1
                for (int i = j + 1 + lane; i < k; i += 32) S[i * k + j] /= sd;
                if (lane == 0) S[j * k + j] = sd;
                __syncwarp();
                #pragma unroll 1
                for (int i = j + 1 + lane; i < k; i += 32) {
                    const double lij = S[i * k + j];
                    #pragma unroll 1
                    for (int c = j + 1; c <= i; ++c) S[i * k + c] = fma(-lij, S[c * k + j], S[i * k + c]);
                }
                __syncwarp();
            }
            bool pass = false, numeric = false, thin = false;
            if (!pd) {
                numeric = true;
            } else {
                // Lambda = -S^-1 V[act]; lane c handles rhs column c (0 = constant term)
                if (lane < t1) {
                    #pragma unroll 1
                    for (int i = 0; i < k; ++i) {
                        double s = -__ldg(P.V + (size_t)act[i] * t1 + lane);
                        #pragma unroll 1
                        for (int j = 0; j < i; ++j) s = fma(-S[i * k + j], Lam[j * t1 + lane], s);
                        Lam[i * t1 + lane] = s / S[i * k + i];
                    }
                    #pragma unroll 1
                    for (int i = k - 1; i >= 0; --i) {
                        double s = Lam[i * t1 + lane];
                        #pragma unroll 1
                        for (int j = i + 1; j < k; ++j) s = fma(-S[j * k + i], Lam[j * t1 + lane], s);
                        Lam[i * t1 + lane] = s / S[i * k + i];
                    }
                }
                __syncwarp();
                // necessary condition (see k34_kkt.cu): every nonzero multiplier row must reach lambda_j(theta) >= 0 in the box
                bool reject = false;
                #pragma unroll 1
                for (int j = lane; j < k; j += 32) {
                    double ub = Lam[j * t1], mx = 0.0, mag = fabs(Lam[j * t1]);
                    #pragma unroll 1
                    for (int c = 0; c < t; ++c) {
                        const double a = Lam[j * t1 + 1 + c];
                        const double lo = __ldg(P.th_lo + c), hi = __ldg(P.th_hi + c);
                        mx = fmax(mx, fabs(a));
                        if (a != 0.0) { const double term = fmax(a * lo, a * hi); ub += term; mag += fabs(term); }
                    }
                    if (mx > PPG_ZERO_ROW) { if (ub < -1e-9 * fmax(1.0, mag)) reject = true; }
                    else if (mx <= PPG_ZERO_ROW && Lam[j * t1] < -PPG_FEAS_TOL) reject = true;   // zero-row rule of the row build, early
                }
                if (__any_sync(PPG_FULL, reject)) {
                    if (use_pre && lane == 0) status[idx] = st;
                    continue;   // not optimal: status keeps PPG_ST_FEAS only
                }
                // region rows into the tableau: [f | a | 1]
                bool zero_viol = false;
                double lo1 = -CUDART_INF, hi1 = CUDART_INF;
                #pragma unroll 1
                for (int row = lane; row < m; row += 32) {
                    double* T = Tab + (size_t)row * lds;
                    if (row < mi) {
                        if (mask_test(mk, row)) {
                            const int pos = mask_rank(mk, row);
                            T[0] = Lam[pos * t1];
                            #pragma unroll 1
                            for (int c = 1; c < t1; ++c) T[c] = -Lam[pos * t1 + c];
                        } else {
                            #pragma unroll 1
                            for (int c = 0; c < t1; ++c) T[c] = __ldg(P.V + (size_t)row * t1 + c);
                            #pragma unroll 1
                            for (int a = 0; a < k; ++a) {
                                // G is symmetric: G[act[a]][row] instead of G[row][act[a]] - consecutive lanes read
                                // consecutive doubles of ONE row of G (8 sectors per warp load instead of 32)
                                const double g = __ldg(P.G + (size_t)act[a] * mi + row);
                                #pragma unroll 1
                                for (int c = 0; c < t1; ++c) T[c] = fma(g, Lam[a * t1 + c], T[c]);
                            }
                            #pragma unroll 1
                            for (int c = 1; c < t1; ++c) T[c] = -T[c];
                        }
                    } else {
                        const int o = row - mi;
                        T[0] = __ldg(P.b_t + o);
                        #pragma unroll 1
                        for (int c = 1; c < t1; ++c) T[c] = __ldg(P.A_t + (size_t)o * t + c - 1);
                    }
                    double mx = 0.0, nn = 0.0;
                    #pragma unroll 1
                    for (int c = 1; c < t1; ++c) { mx = fmax(mx, fabs(T[c])); nn = fma(T[c], T[c], nn); }
                    unsigned char fl = 0;
                    if (!(mx <= PPG_ZERO_ROW)) {
                        const double inv = 1.0 / sqrt(nn);
                        #pragma unroll 1
                        for (int c = 0; c < t1; ++c) T[c] *= inv;
                        T[t1] = 1.0;
                        fl = 1;
                        if (t == 1) { const double q = T[0] / T[1]; if (T[1] > 0.0) hi1 = fmin(hi1, q); else lo1 = fmax(lo1, q); }
                    } else if (T[0] < -PPG_FEAS_TOL) {
                        zero_viol = true;
                    }
                    flag[row] = fl;
                }
                __syncwarp();
                if (!__any_sync(PPG_FULL, zero_viol)) {
                    if (t == 1) {
                        // interval [lo, hi] of the 1-D polytope (get_bounds_1d, mpqp_utils.py:304-315)
#pragma unroll
                        for (int o = 16; o > 0; o >>= 1) {
                            lo1 = fmax(lo1, shfl_xor_d(lo1, o));
                            hi1 = fmin(hi1, shfl_xor_d(hi1, o));
                        }
                        pass = (lo1 + 0.5 * PPG_WIDTH_1D <= hi1);
                    } else {
                        const K4cOut res = k4c_solve(Tab, flag, bvar, alpha, kind, nbv, prow, m, t, lds, PPG_RADIUS_SCREEN, lane);
                        pass = res.code == PPG_LP_EARLY || (res.code == PPG_LP_OPTIMAL && res.beta >= PPG_RADIUS_SCREEN);
                        thin = res.code == PPG_LP_OPTIMAL && !pass && res.beta >= -PPG_RADIUS_BAND;
                        if (res.code == PPG_LP_ITERLIM) numeric = true;
                        n_lp++; n_piv += res.pivots; n_work += (unsigned long long)res.work;
                    }
                }
            }
            if (lane == 0) {
                uint8_t s2 = st;
                if (pass) s2 |= PPG_ST_OPT;
                if (thin) s2 |= PPG_ST_THIN;
                if (numeric) { s2 |= PPG_ST_NUMERIC; n_num++; }
                if (s2 != st || use_pre) status[idx] = s2;
            }
        }
    }
    if (lane == 0 && (n_lp || n_num)) {
        atomicAdd(&counters[CNT_K4_LPS], n_lp);
        atomicAdd(&counters[CNT_K4_PIVOTS], n_piv);
        atomicAdd(&counters[CNT_K4_WORK], n_work);
        if (n_num) atomicAdd(&counters[CNT_NUMERIC], n_num);
    }
}

// returns cudaSuccess with *handled == false when the candidate's scratch does not fit shared memory
cudaError_t launch_k34_compact(const DevProgram& P, const uint64_t* masks, long long n, int k_act, uint8_t* status,
                               unsigned long long* queue, unsigned long long* counters, int sm_count, cudaStream_t st,
                               int use_pre, bool* handled) {
    *handled = false;
    static const int on = getenv("PPGPU_K34_COMPACT") ? atoi(getenv("PPGPU_K34_COMPACT")) : 1;
    if (!on) return cudaSuccess;
    constexpr int WPC = 4;
    const int m = P.R0, t1 = P.t + 1, ld = P.t + 2, lds = ld | 1, k = k_act;
    size_t wb = (size_t)m * lds * 8 + (size_t)k * k * 8 + (size_t)k * t1 * 8 + (size_t)2 * lds * 8 +
                (size_t)(((k + 1) & ~1) + ((m + 1) & ~1) + 2 * ((lds + 1) & ~1)) * 4 + (size_t)m;
    wb = (wb + 15) & ~(size_t)15;
    const size_t smem = wb * WPC;
    if (smem > 200 * 1024) return cudaSuccess;
    cudaError_t e = allow_max_smem(k34c_kernel);
    if (e != cudaSuccess) return e;
    int occ = 0;
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k34c_kernel, 32 * WPC, smem);
    if (e != cudaSuccess) return e;
    if (occ < 1) occ = 1;
    // a warp decides the candidates of a queue item one after another: 32 per item, fewer when the level would leave
    // warps of the resident grid without an item (level 1: 100 candidates were 4 items, 25 candidates in a row per warp)
    const long long warps = (long long)sm_count * occ * WPC;
    const int per_item = (int)std::min<long long>(32, std::max<long long>(1, (n + warps - 1) / warps));
    const long long items = (n + per_item - 1) / per_item;
    long long grid = (long long)sm_count * occ;
    const long long need = (items + WPC - 1) / WPC;
    if (grid > need) grid = need;
    if (grid < 1) grid = 1;
    k34c_kernel<<<(unsigned)grid, 32 * WPC, smem, st>>>(P, masks, n, k_act, status, queue, counters, use_pre, (int)wb, lds,
                                                        per_item);
    *handled = true;
    return cudaGetLastError();
}

// ---- batched Chebyshev balls of arbitrary polytopes {theta : E theta <= f} (chebyshev_ball, utils/chebyshev_ball.py:10-63:
// max r : E_i theta + |E_i| r <= f_i; CriticalRegion.is_full_dimension, critical_region.py:89-105; the constructor's
// warnings(), mplp_program.py:162-215).  One warp per polytope, the LP of k4c_solve on the warp's shared-memory tableau.
__global__ void __launch_bounds__(128)
cheb_batch_kernel(const double* __restrict__ rows, const long long* __restrict__ row_off, long long n_poly, int t,
                  double* __restrict__ radius, int* __restrict__ code, int warp_bytes, int lds, int max_rows) {
    extern __shared__ unsigned char cheb_smem[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, t1 = t + 1;
    unsigned char* base = cheb_smem + (size_t)warp * warp_bytes;
    double* Tab = reinterpret_cast<double*>(base); base += (size_t)max_rows * lds * 8;
    double* alpha = reinterpret_cast<double*>(base); base += (size_t)lds * 8;
    double* prow = reinterpret_cast<double*>(base); base += (size_t)lds * 8;
    int* bvar = reinterpret_cast<int*>(base); base += (size_t)((max_rows + 1) & ~1) * 4;
    int* kind = reinterpret_cast<int*>(base); base += (size_t)((lds + 1) & ~1) * 4;
    int* nbv = reinterpret_cast<int*>(base); base += (size_t)((lds + 1) & ~1) * 4;
    unsigned char* flag = base;
    for (long long p = (long long)blockIdx.x * (blockDim.x >> 5) + warp; p < n_poly; p += (long long)gridDim.x * (blockDim.x >> 5)) {
        const long long r0 = row_off[p];
        const int m = (int)(row_off[p + 1] - r0);
        bool bad = false;
        __syncwarp();
#pragma unroll 1
        for (int i = lane; i < m; i += 32) {
            const double* src = rows + (size_t)(r0 + i) * t1;
            double* T = Tab + (size_t)i * lds;
            double nn = 0.0;
            T[0] = src[0];
#pragma unroll 1
            for (int c = 1; c < t1; ++c) { T[c] = src[c]; nn = fma(src[c], src[c], nn); }
            T[t1] = sqrt(nn);
            // a row without theta reads 0 <= f: either always true (dropped) or never (the polytope is empty)
            flag[i] = nn > 0.0 ? 1 : 0;
            if (!(nn > 0.0) && src[0] < 0.0) bad = true;
        }
        __syncwarp();
        K4cOut res; res.code = PPG_LP_INFEAS_EQ; res.beta = -CUDART_INF;
        if (!__any_sync(PPG_FULL, bad) && m > 0)
            res = k4c_solve(Tab, flag, bvar, alpha, kind, nbv, prow, m, t, lds, CUDART_INF, lane);
        if (lane == 0) { radius[p] = res.beta; code[p] = res.code; }
    }
}

cudaError_t launch_cheb_batch(const double* rows, const long long* row_off, long long n_poly, int t, int max_rows,
                              double* radius, int* code, int sm_count, cudaStream_t st) {
    constexpr int WPC = 4;
    const int ld = t + 2, lds = ld | 1;
    size_t wb = (size_t)max_rows * lds * 8 + (size_t)2 * lds * 8 + (size_t)(((max_rows + 1) & ~1) + 2 * ((lds + 1) & ~1)) * 4 +
                (size_t)max_rows;
    wb = (wb + 15) & ~(size_t)15;
    const size_t smem = wb * WPC;
    if (smem > 200 * 1024) return cudaErrorInvalidValue;
    cudaError_t e = allow_max_smem(cheb_batch_kernel);
    if (e != cudaSuccess) return e;
    long long grid = (n_poly + WPC - 1) / WPC;
    if (grid > (long long)sm_count * 4) grid = (long long)sm_count * 4;
    if (grid < 1) return cudaSuccess;
    cheb_batch_kernel<<<(unsigned)grid, 32 * WPC, smem, st>>>(rows, row_off, n_poly, t, radius, code, (int)wb, lds, max_rows);
    return cudaGetLastError();
}

// ---- K10: batched Chebyshev balls of FACETS {theta : E theta <= f, a_i theta = f_i} (the geometric mpQP algorithm steps across
// every facet of a region from its centre).  theta = theta0 + N z with theta0 = f_i a_i / |a_i|^2 and N the t - 1 columns other
// than k of the Householder reflector H = I - 2 v v' / v'v, v = n + sign(n_k) e_k, n = a_i / |a_i|, k = argmax |n_k|: H is
// symmetric and orthogonal and maps n to -sign(n_k) e_k, so its other columns are an orthonormal basis of the hyperplane and
// |N' a_j| = |P a_j|.  The facet LP is then the Chebyshev LP of {z : (N' a_j) z <= f_j - a_j theta0} in t - 1 variables.

// row j of the polytope in the facet's coordinates: dst = [f_j - a_j theta0 | N' a_j | |N' a_j|]; returns |a_j|
__device__ __forceinline__ double k10_row(const double* __restrict__ src, const double* __restrict__ v, double c2,
                                          const double* __restrict__ th0, int t, int k, double* __restrict__ dst) {
    double s = 0.0, at = 0.0, an = 0.0;
#pragma unroll 1
    for (int c = 0; c < t; ++c) { const double a = src[1 + c]; s = fma(v[c], a, s); at = fma(a, th0[c], at); an = fma(a, a, an); }
    s *= c2;
    double nn = 0.0;
    int o = 1;
#pragma unroll 1
    for (int c = 0; c < t; ++c) {
        if (c == k) continue;
        const double h = fma(-s, v[c], src[1 + c]);
        dst[o++] = h;
        nn = fma(h, h, nn);
    }
    dst[0] = src[0] - at;
    dst[t] = sqrt(nn);
    return sqrt(an);
}

// the per-warp shared-memory layout of K10 (launch_facet_cheb sizes it).  The callees below rebuild it from the warp's base
// pointer instead of taking ten pointers: the kernel then keeps one pointer live across its calls and needs no stack.
struct K10Smem { double *Tab, *alpha, *prow, *v, *th0, *M; int *bvar, *kind, *nbv; unsigned char* flag; };
__device__ __forceinline__ K10Smem k10_smem(unsigned char* base, int max_rows, int lds, int t) {
    K10Smem S;
    S.Tab = reinterpret_cast<double*>(base); base += (size_t)max_rows * lds * 8;
    S.alpha = reinterpret_cast<double*>(base); base += (size_t)lds * 8;
    S.prow = reinterpret_cast<double*>(base); base += (size_t)lds * 8;
    S.v = reinterpret_cast<double*>(base); base += (size_t)t * 8;
    S.th0 = reinterpret_cast<double*>(base); base += (size_t)t * 8;
    S.M = reinterpret_cast<double*>(base); base += (size_t)t * (t + 1) * 8;   // final basis, then its solution
    S.bvar = reinterpret_cast<int*>(base); base += (size_t)((max_rows + 1) & ~1) * 4;
    S.kind = reinterpret_cast<int*>(base); base += (size_t)((lds + 1) & ~1) * 4;
    S.nbv = reinterpret_cast<int*>(base); base += (size_t)((lds + 1) & ~1) * 4;
    S.flag = base;
    return S;
}

__device__ __noinline__ K4cOut k10_lp(unsigned char* base, int max_rows, int lds, int m, int t, int lane) {
    const K10Smem S = k10_smem(base, max_rows, lds, t);
    return k4c_solve(S.Tab, S.flag, S.bvar, S.alpha, S.kind, S.nbv, S.prow, m, t - 1, lds, CUDART_INF, lane);
}

// K10's output for one facet (lane 0): radius and code of the LP, and the centre - the vertex of the final basis.  Every
// nonbasic variable is 0 there: a free one (z_c or r) by itself, a slack because its row is tight.  k4c_solve keeps no row
// for a free basic variable, so the tight rows are rebuilt from the input and the nc x nc system [rhs | z r] is solved by
// Gaussian elimination with partial pivoting.
__device__ __noinline__ void k10_centre(const double* __restrict__ rows, long long r0, int t, int k, double c2, unsigned char* base,
                                        int max_rows, int lds, K4cOut res, double* center, double* radius, int* code) {
    const int t1 = t + 1, nc = t;
    const K10Smem S = k10_smem(base, max_rows, lds, t);
    const double* v = S.v;
    const double* th0 = S.th0;
    const int* nbv = S.nbv;
    double* M = S.M;
    double* th = S.prow;   // k4c_solve's scratch row, free again (lds >= t + 1)
    bool ok = res.code == PPG_LP_OPTIMAL;
    if (ok) {
        const int ldm = nc + 1;
        for (int c = 1; c <= nc; ++c) {
            double* R = M + (size_t)(c - 1) * ldm;
            const int var = nbv[c];
            if (var <= nc) {
                for (int q = 0; q <= nc; ++q) R[q] = 0.0;
                R[var] = 1.0;
            } else {
                k10_row(rows + (size_t)(r0 + var - (nc + 1)) * t1, v, c2, th0, t, k, R);
            }
        }
        for (int c = 1; c <= nc && ok; ++c) {
            int piv = c - 1;
            for (int r = c; r < nc; ++r) if (fabs(M[r * ldm + c]) > fabs(M[piv * ldm + c])) piv = r;
            const double d = M[piv * ldm + c];
            if (!(fabs(d) > 0.0)) { ok = false; break; }
            if (piv != c - 1)
                for (int q = 0; q <= nc; ++q) { const double x = M[(c - 1) * ldm + q]; M[(c - 1) * ldm + q] = M[piv * ldm + q]; M[piv * ldm + q] = x; }
            for (int r = c; r < nc; ++r) {
                const double f = M[r * ldm + c] / d;
                for (int q = 0; q <= nc; ++q) M[r * ldm + q] = fma(-f, M[(c - 1) * ldm + q], M[r * ldm + q]);
            }
        }
        if (ok) {
            // back substitution: the solution of variable c - 1 replaces the right-hand side of row c - 1
            for (int c = nc; c >= 1; --c) {
                double s = M[(c - 1) * ldm];
                for (int q = c + 1; q <= nc; ++q) s = fma(-M[(c - 1) * ldm + q], M[(q - 1) * ldm], s);
                M[(c - 1) * ldm] = s / M[(c - 1) * ldm + c];
            }
            // theta = theta0 + H w, w = z placed on the coordinates other than k
            double s = 0.0;
            for (int c = 0, o = 0; c < t; ++c) { th[c] = (c == k) ? 0.0 : M[(o++) * ldm]; s = fma(v[c], th[c], s); }
            s *= c2;
            for (int c = 0; c < t; ++c) th[c] = th0[c] + fma(-s, v[c], th[c]);
        }
    }
    for (int c = 0; c < t; ++c) center[c] = ok ? th[c] : CUDART_NAN;
    *radius = res.beta;
    *code = res.code;
}

__global__ void __launch_bounds__(128)
facet_cheb_kernel(const double* __restrict__ rows, const long long* __restrict__ row_off, long long n_poly, int t,
                  const long long* __restrict__ facets, long long n_facets, double* __restrict__ center,
                  double* __restrict__ radius, int* __restrict__ code, int warp_bytes, int lds, int max_rows) {
    extern __shared__ unsigned char facet_smem[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, t1 = t + 1;
    unsigned char* const wbase = facet_smem + (size_t)warp * warp_bytes;
    const K10Smem S = k10_smem(wbase, max_rows, lds, t);
    double* Tab = S.Tab;
    double* v = S.v;
    double* th0 = S.th0;
    unsigned char* flag = S.flag;
    for (long long p = (long long)blockIdx.x * (blockDim.x >> 5) + warp; p < n_facets; p += (long long)gridDim.x * (blockDim.x >> 5)) {
        const long long poly = facets[2 * p], fi = facets[2 * p + 1];
        long long r0 = 0;
        int m = 0;
        if (poly >= 0 && poly < n_poly) { r0 = row_off[poly]; m = (int)(row_off[poly + 1] - r0); }
        if (fi < 0 || fi >= m) {   // not a row of a polytope of the batch
            if (lane < t) center[p * t + lane] = CUDART_NAN;
            if (lane == 0) { radius[p] = CUDART_NAN; code[p] = -1; }
            continue;
        }
        const double* src_i = rows + (size_t)(r0 + fi) * t1;
        int k = 0;
        double c2 = 0.0, ai2 = 0.0;
        __syncwarp();
        if (lane == 0) {
            double big = -1.0;
            for (int c = 0; c < t; ++c) { const double a = src_i[1 + c]; ai2 = fma(a, a, ai2); if (fabs(a) > big) { big = fabs(a); k = c; } }
            if (ai2 > 0.0) {
                const double inv = 1.0 / sqrt(ai2), q = src_i[0] / ai2;
                double vv = 0.0;
                for (int c = 0; c < t; ++c) {
                    const double nc_ = src_i[1 + c] * inv;
                    v[c] = nc_ + (c == k ? (nc_ >= 0.0 ? 1.0 : -1.0) : 0.0);
                    vv = fma(v[c], v[c], vv);
                    th0[c] = src_i[1 + c] * q;
                }
                c2 = 2.0 / vv;
            }
        }
        k = __shfl_sync(PPG_FULL, k, 0);
        c2 = shfl_d(c2, 0);
        ai2 = shfl_d(ai2, 0);
        __syncwarp();
        K4cOut res; res.code = PPG_LP_INFEAS_EQ; res.beta = -CUDART_INF;
        bool bad = !(ai2 > 0.0);   // a zero row has no facet
        if (!bad && t == 1) {
            // the facet is the point f_i / a_i: unbounded when every other row holds there, empty otherwise
#pragma unroll 1
            for (int j = lane; j < m; j += 32) {
                const double* src = rows + (size_t)(r0 + j) * t1;
                if (j != fi && src[0] - src[1] * th0[0] < -PPG_HARRIS * fmax(1.0, fabs(src[0]))) bad = true;
            }
            bad = __any_sync(PPG_FULL, bad);
            if (!bad) { res.code = PPG_LP_UNBOUNDED; res.beta = CUDART_INF; }
            if (lane == 0) center[p] = bad ? CUDART_NAN : th0[0];
            if (lane == 0) { radius[p] = res.beta; code[p] = res.code; }
            continue;
        }
        if (!bad) {
#pragma unroll 1
            for (int j = lane; j < m; j += 32) {
                double* T = Tab + (size_t)j * lds;
                const double* src = rows + (size_t)(r0 + j) * t1;
                const double an = k10_row(src, v, c2, th0, t, k, T);
                // a row parallel to the facet is constant on its hyperplane: dropped when it holds there, else the facet is
                // empty.  "Parallel" up to 1e-9 |a_j|: below that the rounding of f_j - a_j theta0 (|f_j| 1e-16), divided by
                // |N' a_j| when the row is scaled, would decide the radius (a facet of radius 3e-6 came out empty)
                const bool live = j != fi && T[t] > PPG_HARRIS * an;
                if (live) {
                    // unit rows: k4c_solve's first pivot (r enters on the row of smallest right-hand side) leaves every
                    // slack >= 0 only when every row's r coefficient is the same
                    const double inv = 1.0 / T[t];
#pragma unroll 1
                    for (int c = 0; c < t; ++c) T[c] *= inv;
                    T[t] = 1.0;
                }
                flag[j] = live ? 1 : 0;
                if (!live && j != fi && T[0] < -PPG_HARRIS * fmax(1.0, fabs(src[0]))) bad = true;
            }
            __syncwarp();
            bad = __any_sync(PPG_FULL, bad);
            if (!bad) res = k10_lp(wbase, max_rows, lds, m, t, lane);
        }
        __syncwarp();
        if (lane == 0) k10_centre(rows, r0, t, k, c2, wbase, max_rows, lds, res, center + p * t, radius + p, code + p);
    }
}

cudaError_t launch_facet_cheb(const double* rows, const long long* row_off, long long n_poly, int t, int max_rows,
                              const long long* facets, long long n_facets, double* center, double* radius, int* code,
                              int sm_count, cudaStream_t st) {
    constexpr int WPC = 4;
    const int ld = t + 1, lds = ld | 1;   // t - 1 variables z, then r
    size_t wb = (size_t)max_rows * lds * 8 + (size_t)2 * lds * 8 + (size_t)2 * t * 8 + (size_t)t * (t + 1) * 8 +
                (size_t)(((max_rows + 1) & ~1) + 2 * ((lds + 1) & ~1)) * 4 + (size_t)max_rows;
    wb = (wb + 15) & ~(size_t)15;
    const size_t smem = wb * WPC;
    if (smem > 200 * 1024) return cudaErrorInvalidValue;
    cudaError_t e = allow_max_smem(facet_cheb_kernel);
    if (e != cudaSuccess) return e;
    long long grid = (n_facets + WPC - 1) / WPC;
    if (grid > (long long)sm_count * 4) grid = (long long)sm_count * 4;
    if (grid < 1) return cudaSuccess;
    facet_cheb_kernel<<<(unsigned)grid, 32 * WPC, smem, st>>>(rows, row_off, n_poly, t, facets, n_facets, center, radius, code,
                                                              (int)wb, lds, max_rows);
    return cudaGetLastError();
}

}  // namespace ppgpu
