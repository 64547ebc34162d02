// K5 - critical-region emission for the candidates that passed the optimality screen. One CTA per region.
//
// Reference work replaced (per region): gen_cr_from_active_set / gen_cr_from_active_set_1d
// (/root/reference/src/ppopt/utils/mpqp_utils.py:89-301):
//   1. optimal_control_law: LU (partial pivoting) of the KKT matrix [[A_act 0],[Q A_act']] with rhs
//      [b_act | F_act ; -c | -H]  (mpqp_program.py:182-190; for an mpLP Q = 0 and the system is the square
//      A_act x = b_act + F_act theta, mplp_program.py:387-395) -> x(theta), lambda(theta)
//   2. rows [-C_ineq ; A_inact A_x - F_inact ; A_t] in THAT order, zero-row filter (atol 1e-8), L2 normalisation
//   3. full-dimension test: Chebyshev radius > 1e-8 (1-D: min + 1e-8 <= max)
//   4. one redundancy LP per kept row (row forced to equality)      (mpqp_utils.py:143-178)
//   5. exact-duplicate removal keeping the first occurrence         (constraint_utilities.py:125-134)
// Output per region: laws (n+k) x (t+1) [const | theta], rows R0 x (t+1) [f | a] normalised, int flags per row
// (bit0 nonzero, bit1 non-redundant, bit2 duplicate of an earlier kept row) and info[4] = {region?, radius, lo, hi}.
//
// Three launches (t > 1):
//   K5a k5_emit_kernel<.., false>  one CTA per region: steps 1-3 (t == 1: all five, the redundancy test is interval arithmetic)
//   K5b k5_redund_kernel           step 4 as ONE batch of (region, row) LPs, one warp per LP, from the rows K5a wrote
//   K5c k5_dedupe_kernel           step 5, one warp per region
// A region's redundancy LPs are independent of each other, but inside one CTA four warps solve the ~110 LPs of a region
// one after another, at the 222 registers of the LU + Chebyshev kernel (2 CTAs per SM).  K5b holds only the LP, runs 4x
// more warps per SM and spreads the LPs of all regions over the whole device.  Every LP is the same routine on the same
// registers as before, so laws, rows, flags, info, status and counters are bit-identical to the fused kernel
// (k5_emit_kernel<.., true>, selected with PPGPU_K5_FUSED=1).
#include <cstdlib>

#include "common.cuh"
#include "launch.h"
#include "lp_core.cuh"

namespace ppgpu {

constexpr int K5_WARPS = 4;
constexpr int K5_THREADS = K5_WARPS * 32;

template <int RPT, int DC, bool FUSED>
__global__ void __launch_bounds__(K5_THREADS)
k5_emit_kernel(DevProgram P, const uint64_t* __restrict__ masks, const long long* __restrict__ sel, long long n_sel,
               int k_act, double* __restrict__ laws_out, double* __restrict__ rows_out, int32_t* __restrict__ flags_out,
               double* __restrict__ info_out, uint8_t* __restrict__ status, unsigned long long* __restrict__ counters) {
    typedef LpCore<1, RPT, DC> Core;
    extern __shared__ double dyn_smem[];
    __shared__ typename Core::Shared sh_all[K5_WARPS];
    __shared__ double red_v[K5_WARPS];
    __shared__ int red_i[K5_WARPS];
    __shared__ double s_info[4];
    __shared__ int s_ok;    // KKT solved and no zero row with negative rhs
    __shared__ int s_full;  // full-dimension test passed
    __shared__ int s_thin;  // ... with a radius inside PPG_RADIUS_BAND of the threshold
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int n = P.n, t = P.t, t1 = P.t + 1, m = P.m, ne = P.ne, mi = P.mi, R0 = P.R0, W = P.W;
    const int k = ne + k_act, N = n + k, ld = N + t1;
    double* M = dyn_smem;                                  // N x ld
    double* rows = M + (size_t)N * ld;                     // R0 x t1
    int* flags = reinterpret_cast<int*>(rows + (size_t)R0 * t1);  // R0
    int* actf = flags + R0;                                // k
    int* keptf = actf + k;                                 // R0: redundancy verdicts (merged into flags after a barrier)
    unsigned long long n_lp = 0, n_piv = 0, n_work = 0;

    for (long long si = blockIdx.x; si < n_sel; si += gridDim.x) {
        const long long idx = sel[si];
        const uint64_t* mk = masks + idx * W;
        __syncthreads();
        for (int j = tid; j < k; j += K5_THREADS) actf[j] = j < ne ? j : ne + mask_nth(mk, W, j - ne);
        if (tid == 0) { s_ok = 1; s_full = 0; s_thin = 0; s_info[0] = 0.0; s_info[1] = -CUDART_INF; s_info[2] = -CUDART_INF; s_info[3] = CUDART_INF; }
        __syncthreads();
        // ---- KKT matrix
        for (int e = tid; e < N * ld; e += K5_THREADS) {
            const int r = e / ld, c = e - r * ld;
            double v = 0.0;
            if (r < k) {
                const int row = actf[r];
                if (c < n) v = __ldg(P.A + (size_t)row * n + c);
                else if (c == N) v = __ldg(P.b + row);
                else if (c > N) v = __ldg(P.F + (size_t)row * t + (c - N - 1));
            } else {
                const int i = r - k;
                if (c < n) v = __ldg(P.Q + (size_t)i * n + c);
                else if (c < N) v = __ldg(P.A + (size_t)actf[c - n] * n + i);
                else if (c == N) v = -__ldg(P.c + i);
                else v = -__ldg(P.H + (size_t)i * t + (c - N - 1));
            }
            M[e] = v;
        }
        __syncthreads();
        // ---- LU with partial pivoting (first maximal entry wins ties)
        for (int col = 0; col < N; ++col) {
            double best = -1.0; int p = 0x7fffffff;
            for (int i = col + tid; i < N; i += K5_THREADS) {
                const double a = fabs(M[(size_t)i * ld + col]);
                if (a > best) { best = a; p = i; }
            }
            warp_argmax(best, p);
            if (lane == 0) { red_v[warp] = best; red_i[warp] = p; }
            __syncthreads();
            best = red_v[0]; p = red_i[0];
#pragma unroll
            for (int w = 1; w < K5_WARPS; ++w)
                if (red_v[w] > best || (red_v[w] == best && red_i[w] < p)) { best = red_v[w]; p = red_i[w]; }
            if (!(best > 0.0) || !isfinite(best)) { if (tid == 0) s_ok = 0; __syncthreads(); break; }
            if (p != col) {
                for (int c = tid; c < ld; c += K5_THREADS) {
                    const double a = M[(size_t)p * ld + c];
                    M[(size_t)p * ld + c] = M[(size_t)col * ld + c];
                    M[(size_t)col * ld + c] = a;
                }
            }
            __syncthreads();
            const double inv = 1.0 / M[(size_t)col * ld + col];
            __syncthreads();
            for (int i = col + 1 + tid; i < N; i += K5_THREADS) M[(size_t)i * ld + col] *= inv;
            __syncthreads();
            const int tw = ld - col - 1, th = N - col - 1;
            for (int e = tid; e < tw * th; e += K5_THREADS) {
                const int i = col + 1 + e / tw, c = col + 1 + e % tw;
                M[(size_t)i * ld + c] = fma(-M[(size_t)i * ld + col], M[(size_t)col * ld + c], M[(size_t)i * ld + c]);
            }
            __syncthreads();
        }
        __syncthreads();
        const bool singular = s_ok == 0;
        if (!singular) {
            if (tid < t1) {
                const int c = tid;
                for (int i = N - 1; i >= 0; --i) {
                    double s = M[(size_t)i * ld + N + c];
                    for (int j = i + 1; j < N; ++j) s = fma(-M[(size_t)i * ld + j], M[(size_t)j * ld + N + c], s);
                    M[(size_t)i * ld + N + c] = s / M[(size_t)i * ld + i];
                }
            }
            __syncthreads();
            for (int e = tid; e < N * t1; e += K5_THREADS) {
                const int i = e / t1, c = e - i * t1;
                laws_out[(size_t)si * N * t1 + e] = M[(size_t)i * ld + N + c];
            }
            // ---- region rows in the reference order, zero filter, normalisation
            const int n_inact = mi - k_act;
            for (int r0 = tid; r0 < m + P.q; r0 += K5_THREADS) {
                int r = -1;
                double v[DC];
#pragma unroll
                for (int c = 0; c < DC; ++c) v[c] = 0.0;
                if (r0 < m) {
                    const int i = r0;
                    if (i >= ne) {
                        const int bi = i - ne;
                        const int rk = mask_rank(mk, bi);
                        if (mask_test(mk, bi)) {
                            r = rk;
                            const double* l = M + (size_t)(n + ne + rk) * ld + N;
#pragma unroll
                            for (int c = 0; c < DC; ++c)
                                if (c < t1) v[c] = c == 0 ? l[0] : -l[c];
                        } else {
                            r = k_act + (bi - rk);
                            for (int j = 0; j < n; ++j) {
                                const double a = __ldg(P.A + (size_t)i * n + j);
#pragma unroll
                                for (int c = 0; c < DC; ++c)
                                    if (c < t1) v[c] = fma(a, M[(size_t)j * ld + N + c], v[c]);
                            }
#pragma unroll
                            for (int c = 0; c < DC; ++c)
                                if (c < t1) v[c] = c == 0 ? __ldg(P.b + i) - v[0] : v[c] - __ldg(P.F + (size_t)i * t + c - 1);
                        }
                    }
                } else {
                    const int o = r0 - m;
                    r = k_act + n_inact + o;
                    v[0] = __ldg(P.b_t + o);
#pragma unroll
                    for (int c = 1; c < DC; ++c)
                        if (c < t1) v[c] = __ldg(P.A_t + (size_t)o * t + c - 1);
                }
                if (r >= 0) {
                    double mx = 0.0, nn = 0.0;
#pragma unroll
                    for (int c = 1; c < DC; ++c)
                        if (c < t1) { mx = fmax(mx, fabs(v[c])); nn = fma(v[c], v[c], nn); }
                    int fl = 0;
                    if (!(mx <= PPG_ZERO_ROW)) {
                        fl = 1;
                        const double inv = 1.0 / sqrt(nn);
#pragma unroll
                        for (int c = 0; c < DC; ++c) v[c] *= inv;
                    } else if (v[0] < -PPG_FEAS_TOL) {
                        atomicExch(&s_ok, 0);  // zero row with negative rhs: not optimal
                    }
                    flags[r] = fl;
                    keptf[r] = 0;
#pragma unroll
                    for (int c = 0; c < DC; ++c)
                        if (c < t1) rows[(size_t)r * t1 + c] = v[c];
                }
            }
        }
        __syncthreads();
        bool region = !singular && s_ok != 0;
        // ---- full-dimension test (warp 0)
        if (region) {
            if (warp == 0) {
                if (t == 1) {
                    double lo = -CUDART_INF, hi = CUDART_INF;
                    for (int r = lane; r < R0; r += 32)
                        if (flags[r] & 1) {
                            const double q = rows[(size_t)r * 2] / rows[(size_t)r * 2 + 1];
                            if (rows[(size_t)r * 2 + 1] > 0.0) hi = fmin(hi, q); else lo = fmax(lo, q);
                        }
#pragma unroll
                    for (int o = 16; o > 0; o >>= 1) {
                        lo = fmax(lo, shfl_xor_d(lo, o));
                        hi = fmin(hi, shfl_xor_d(hi, o));
                    }
                    if (lane == 0) {
                        s_info[1] = 0.5 * (hi - lo); s_info[2] = lo; s_info[3] = hi;
                        s_full = (lo + PPG_WIDTH_1D <= hi) ? 1 : 0;
                    }
                } else {
                    // Chebyshev LP, then the radius of the LP's own point re-evaluated on the untouched rows: the simplex
                    // relaxes rows by up to 1e-9 per pivot (Harris bound, snapping), so its beta is an UPPER bound of the
                    // radius and min_i (f_i - a_i theta*) a LOWER one; the decision uses the lower bound.  An early exit
                    // whose point does not clear the band is repeated without early exit (attempt 1).
                    double rad_lo = -CUDART_INF, rad_hi = -CUDART_INF;
                    int code = PPG_LP_OPTIMAL;
                    for (int attempt = 0; attempt < 2; ++attempt) {
                        double T[RPT][DC];
                        int rflag[RPT], bv[RPT];
                        static_for<RPT>([&](auto RR) {
                            constexpr int rr = decltype(RR)::value;
                            const int row = rr * 32 + lane;
                            const bool on = row < R0 && (flags[row] & 1);
#pragma unroll
                            for (int c = 0; c < DC; ++c) T[rr][c] = (on && c < t1) ? rows[(size_t)row * t1 + c] : ((on && c == t1) ? 1.0 : 0.0);
                            rflag[rr] = on ? 1 : 0;
                            bv[rr] = 0;
                        });
                        const double thr = attempt == 0 ? PPG_RADIUS + PPG_RADIUS_BAND : CUDART_INF;
                        LpOut res = Core::solve(sh_all[0], T, rflag, R0, t1, thr, true, lane, true, &bv);
                        n_lp++; n_piv += res.pivots; n_work += (unsigned long long)res.work;
                        code = res.code;
                        rad_hi = res.beta;
                        if (code != PPG_LP_EARLY && code != PPG_LP_OPTIMAL) break;
                        // theta* from the rows of the basic free variables (nonbasic ones sit at 0)
                        double* th = &sh_all[0].P[0][0][0];   // scratch: the LP is over
                        __syncwarp();
                        if (lane < t) th[lane] = 0.0;
                        __syncwarp();
                        static_for<RPT>([&](auto RR) {
                            constexpr int rr = decltype(RR)::value;
                            if (rflag[rr] == 3) {
                                const int c = bv[rr] < 0 ? -bv[rr] : bv[rr];
                                if (c >= 1 && c <= t) th[c - 1] = bv[rr] < 0 ? -T[rr][0] : T[rr][0];
                            }
                        });
                        __syncwarp();
                        double lo = CUDART_INF;
                        for (int r = lane; r < R0; r += 32)
                            if (flags[r] & 1) {
                                double sl = rows[(size_t)r * t1];
                                for (int c = 0; c < t; ++c) sl = fma(-rows[(size_t)r * t1 + 1 + c], th[c], sl);
                                lo = fmin(lo, sl);
                            }
#pragma unroll
                        for (int o = 16; o > 0; o >>= 1) lo = fmin(lo, shfl_xor_d(lo, o));
                        rad_lo = lo;
                        __syncwarp();
                        if (code == PPG_LP_OPTIMAL || rad_lo > PPG_RADIUS + PPG_RADIUS_BAND) break;
                    }
                    const bool solved = code == PPG_LP_EARLY || code == PPG_LP_OPTIMAL;
                    const bool ok = solved && rad_lo > PPG_RADIUS;
                    if (lane == 0) {
                        s_info[1] = solved ? rad_lo : rad_hi;
                        s_full = ok ? 1 : 0;
                        s_thin = (solved && rad_hi >= -PPG_RADIUS_BAND && rad_lo <= PPG_RADIUS + PPG_RADIUS_BAND) ? 1 : 0;
                    }
                }
            }
            __syncthreads();
            region = s_full != 0;
        }
        // ---- redundancy tests
        if (region) {
            if (t == 1) {
                const double lo = s_info[2], hi = s_info[3];
                for (int r = tid; r < R0; r += K5_THREADS)
                    if (flags[r] & 1) {
                        const double q = rows[(size_t)r * 2] / rows[(size_t)r * 2 + 1];
                        if (lo <= q && q <= hi) keptf[r] = 1;
                    }
            } else if constexpr (FUSED) {
                for (int a = warp; a < R0; a += K5_WARPS) {
                    if (!(flags[a] & 1)) continue;
                    double T[RPT][DC];
                    int rflag[RPT];
                    static_for<RPT>([&](auto RR) {
                        constexpr int rr = decltype(RR)::value;
                        const int row = rr * 32 + lane;
                        const bool on = row < R0 && (flags[row] & 1);
#pragma unroll
                        for (int c = 0; c < DC; ++c)
                            T[rr][c] = (on && c < t1) ? rows[(size_t)row * t1 + c] : ((on && c == t1 && row != a) ? 1.0 : 0.0);
                        rflag[rr] = on ? (row == a ? 2 : 1) : 0;
                    });
                    LpOut res = Core::solve(sh_all[warp], T, rflag, R0, t1, -PPG_REDUND_TOL, false, lane);
                    n_lp++; n_piv += res.pivots; n_work += (unsigned long long)res.work;
                    const bool feas = res.code == PPG_LP_EARLY || res.code == PPG_LP_UNBOUNDED ||
                                      (res.code == PPG_LP_OPTIMAL && res.beta >= -PPG_REDUND_TOL);
                    if (lane == 0 && feas) keptf[a] = 1;
                }
            }
            __syncthreads();
            for (int r = tid; r < R0; r += K5_THREADS) if (keptf[r]) flags[r] |= 2;
            __syncthreads();
            if (FUSED && t != 1) {
                // duplicates among kept rows (value equality, first occurrence survives); verdicts land after a barrier
                for (int i = tid; i < R0; i += K5_THREADS) {
                    bool dup = false;
                    if ((flags[i] & 3) == 3) {
                        for (int j = 0; j < i && !dup; ++j) {
                            if ((flags[j] & 3) != 3) continue;
                            bool same = true;
                            for (int c = 0; c < t1 && same; ++c) same = rows[(size_t)i * t1 + c] == rows[(size_t)j * t1 + c];
                            dup = same;
                        }
                    }
                    keptf[i] = dup ? 1 : 0;
                }
                __syncthreads();
                for (int r = tid; r < R0; r += K5_THREADS) if (keptf[r]) flags[r] |= 4;
            }
            __syncthreads();
        }
        // ---- outputs
        for (int e = tid; e < R0 * t1; e += K5_THREADS) rows_out[(size_t)si * R0 * t1 + e] = singular ? 0.0 : rows[e];
        for (int r = tid; r < R0; r += K5_THREADS) flags_out[(size_t)si * R0 + r] = singular ? 0 : flags[r];
        if (tid == 0) {
            info_out[si * 4 + 0] = region ? 1.0 : (singular ? -1.0 : 0.0);
            info_out[si * 4 + 1] = s_info[1];
            info_out[si * 4 + 2] = s_info[2];
            info_out[si * 4 + 3] = s_info[3];
            uint8_t st = status[idx];
            if (region) st |= PPG_ST_REGION;
            if (s_thin && !singular) st |= PPG_ST_THIN;
            if (singular) st |= PPG_ST_NUMERIC;
            status[idx] = st;
        }
    }
    if (lane == 0 && n_lp) {
        atomicAdd(&counters[CNT_K5_LPS], n_lp);
        atomicAdd(&counters[CNT_K5_PIVOTS], n_piv);
        atomicAdd(&counters[CNT_K5_WORK], n_work);
    }
}

// K5b: the redundancy LPs of every region of the launch as one flat list of (region, row) pairs, pair = si * R0 + row.
// Warps take K5B_CHUNK consecutive pairs at a time from an atomic queue (consecutive warps work on the same region, whose
// rows then come from L1 / L2); pairs of a non-region or of a zero row are dropped without an LP.  The LP, its tableau and
// the verdict rule are those of the fused kernel.  The verdict lands in bit 1 of the row's flag word, which no other warp
// of the launch writes (bit 0, the only bit read here, never changes).
constexpr int K5B_WARPS = 4;
constexpr int K5B_CHUNK = 4;

// CTAs per SM the register budget is planned for, by tableau doubles a lane: <= 16: 4 (16 warps, <= 128 registers a thread);
// 32: 3 (<= 168; at 128 the bench instance <4, 8> spills); 64: 2; 128 (<8, 16>): 1, where the tableau alone needs 256
template <int RPT, int DC>
constexpr int k5b_min_ctas() { return RPT * DC <= 16 ? 4 : (RPT * DC <= 32 ? 3 : (RPT * DC <= 64 ? 2 : 1)); }

template <int RPT, int DC>
__global__ void __launch_bounds__(K5B_WARPS * 32, k5b_min_ctas<RPT, DC>())
k5_redund_kernel(int R0, int t1, long long n_sel, const double* __restrict__ rows_out, int32_t* flags_out,
                 const double* __restrict__ info_out, unsigned long long* __restrict__ queue,
                 unsigned long long* __restrict__ counters) {
    typedef LpCore<1, RPT, DC> Core;
    __shared__ typename Core::Shared sh_all[K5B_WARPS];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const long long n_pairs = n_sel * R0;
    unsigned long long n_lp = 0, n_piv = 0, n_work = 0;
    for (;;) {
        unsigned long long v = 0;
        if (lane == 0) v = atomicAdd(queue, (unsigned long long)K5B_CHUNK);
        const long long base = (long long)__shfl_sync(PPG_FULL, v, 0);
        if (base >= n_pairs) break;
        bool live = false;
        if (lane < K5B_CHUNK && base + lane < n_pairs) {
            const long long pr = base + lane;
            live = __ldg(info_out + (pr / R0) * 4) == 1.0 && (flags_out[pr] & 1);
        }
        unsigned todo = __ballot_sync(PPG_FULL, live);
        while (todo) {
            const int src = __ffs((int)todo) - 1;
            todo &= todo - 1u;
            const long long pr = base + src, si = pr / R0;
            const int a = (int)(pr - si * R0);
            const double* rows = rows_out + (size_t)si * R0 * t1;
            const int32_t* flags = flags_out + (size_t)si * R0;
            double T[RPT][DC];
            int rflag[RPT];
            static_for<RPT>([&](auto RR) {
                constexpr int rr = decltype(RR)::value;
                const int row = rr * 32 + lane;
                const bool on = row < R0 && (flags[row] & 1);
#pragma unroll
                for (int c = 0; c < DC; ++c)
                    T[rr][c] = (on && c < t1) ? __ldg(rows + (size_t)row * t1 + c) : ((on && c == t1 && row != a) ? 1.0 : 0.0);
                rflag[rr] = on ? (row == a ? 2 : 1) : 0;
            });
            LpOut res = Core::solve(sh_all[warp], T, rflag, R0, t1, -PPG_REDUND_TOL, false, lane);
            n_lp++; n_piv += res.pivots; n_work += (unsigned long long)res.work;
            const bool feas = res.code == PPG_LP_EARLY || res.code == PPG_LP_UNBOUNDED ||
                              (res.code == PPG_LP_OPTIMAL && res.beta >= -PPG_REDUND_TOL);
            if (lane == 0 && feas) atomicOr(flags_out + pr, 2);
        }
    }
    if (lane == 0 && n_lp) {
        atomicAdd(&counters[CNT_K5_LPS], n_lp);
        atomicAdd(&counters[CNT_K5_PIVOTS], n_piv);
        atomicAdd(&counters[CNT_K5_WORK], n_work);
    }
}

// K5c: exact duplicates among the kept rows of a region (value equality, the first occurrence survives), one warp per region.
// A row's verdict is taken before any bit 2 of the region is written.
constexpr int K5C_WARPS = 4;

__global__ void __launch_bounds__(K5C_WARPS * 32)
k5_dedupe_kernel(int R0, int t1, long long n_sel, const double* __restrict__ rows_out, int32_t* __restrict__ flags_out,
                 const double* __restrict__ info_out) {
    const int lane = threadIdx.x & 31;
    const long long nw = (long long)gridDim.x * K5C_WARPS;
    for (long long si = (long long)blockIdx.x * K5C_WARPS + (threadIdx.x >> 5); si < n_sel; si += nw) {
        if (__ldg(info_out + si * 4) != 1.0) continue;
        const double* rows = rows_out + (size_t)si * R0 * t1;
        int32_t* flags = flags_out + (size_t)si * R0;
        unsigned dup = 0;   // bit q: row lane + 32 q
        for (int i = lane, q = 0; i < R0; i += 32, ++q) {
            if ((flags[i] & 3) != 3) continue;
            bool d = false;
            for (int j = 0; j < i && !d; ++j) {
                if ((flags[j] & 3) != 3) continue;
                bool same = true;
                for (int c = 0; c < t1 && same; ++c) same = __ldg(rows + (size_t)i * t1 + c) == __ldg(rows + (size_t)j * t1 + c);
                d = same;
            }
            if (d) dup |= 1u << q;
        }
        __syncwarp();
        for (int i = lane, q = 0; i < R0; i += 32, ++q)
            if ((dup >> q) & 1u) flags[i] |= 4;
    }
}

// PPGPU_K5_FUSED=1: the fused one-CTA-per-region kernel (the A/B reference of the three launches)
static bool k5_fused() {
    static const bool on = getenv("PPGPU_K5_FUSED") && atoi(getenv("PPGPU_K5_FUSED")) != 0;
    return on;
}

int k5_launches(int t) { return k5_fused() || t == 1 ? 1 : 3; }

template <int RPT, int DC>
static cudaError_t launch_k5_t(const DevProgram& P, const uint64_t* masks, const long long* idx, long long n_sel, int k_act,
                               double* laws, double* rows, int32_t* flags, double* info, uint8_t* status,
                               unsigned long long* queue, unsigned long long* counters, int sm_count, cudaStream_t st) {
    const bool fused = k5_fused();
    auto kern = fused ? k5_emit_kernel<RPT, DC, true> : k5_emit_kernel<RPT, DC, false>;
    const int k = P.ne + k_act, N = P.n + k, ld = N + P.t + 1;
    const size_t smem = ((size_t)N * ld + (size_t)P.R0 * (P.t + 1)) * sizeof(double) + (size_t)(2 * P.R0 + k + 2) * sizeof(int);
    if (smem > 200 * 1024) return cudaErrorInvalidValue;
    cudaError_t e;
    if ((e = fit_smem(kern, smem)) != cudaSuccess) return e;
    long long grid = n_sel;
    const long long cap = (long long)sm_count * 8;
    if (grid > cap) grid = cap;
    if (grid < 1) return cudaSuccess;
    kern<<<(unsigned)grid, K5_THREADS, smem, st>>>(P, masks, idx, n_sel, k_act, laws, rows, flags, info, status, counters);
    if ((e = cudaGetLastError()) != cudaSuccess || fused || P.t == 1) return e;

    auto kb = k5_redund_kernel<RPT, DC>;
    if ((e = fit_smem(kb, 0)) != cudaSuccess) return e;
    int occ = 0;
    if ((e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kb, K5B_WARPS * 32, 0)) != cudaSuccess) return e;
    if (occ < 1) occ = 1;
    const long long items = (n_sel * P.R0 + K5B_CHUNK - 1) / K5B_CHUNK;
    grid = (items + K5B_WARPS - 1) / K5B_WARPS;
    if (grid > (long long)sm_count * occ) grid = (long long)sm_count * occ;
    kb<<<(unsigned)grid, K5B_WARPS * 32, 0, st>>>(P.R0, P.t + 1, n_sel, rows, flags, info, queue, counters);
    if ((e = cudaGetLastError()) != cudaSuccess) return e;

    if ((e = fit_smem(k5_dedupe_kernel, 0)) != cudaSuccess) return e;
    grid = (n_sel + K5C_WARPS - 1) / K5C_WARPS;
    if (grid > (long long)sm_count * 16) grid = (long long)sm_count * 16;
    k5_dedupe_kernel<<<(unsigned)grid, K5C_WARPS * 32, 0, st>>>(P.R0, P.t + 1, n_sel, rows, flags, info);
    return cudaGetLastError();
}

#define K5_RPT_SWITCH(DCV)                                                                                                                   \
    if (P.R0 <= 32) return launch_k5_t<1, DCV>(P, masks, idx, n_sel, k_act, laws, rows, flags, info, status, queue, counters, sm_count, st);  \
    if (P.R0 <= 64) return launch_k5_t<2, DCV>(P, masks, idx, n_sel, k_act, laws, rows, flags, info, status, queue, counters, sm_count, st);  \
    if (P.R0 <= 128) return launch_k5_t<4, DCV>(P, masks, idx, n_sel, k_act, laws, rows, flags, info, status, queue, counters, sm_count, st); \
    if (P.R0 <= 256) return launch_k5_t<8, DCV>(P, masks, idx, n_sel, k_act, laws, rows, flags, info, status, queue, counters, sm_count, st); \
    return cudaErrorInvalidValue;

cudaError_t launch_k5(const DevProgram& P, const uint64_t* masks, const long long* idx, long long n_sel, int k_act,
                      double* laws, double* rows, int32_t* flags, double* info, uint8_t* status,
                      unsigned long long* queue, unsigned long long* counters, int sm_count, cudaStream_t st) {
    if (P.t + 2 <= 8) { K5_RPT_SWITCH(8) }
    if (P.t + 2 <= 16) { K5_RPT_SWITCH(16) }
    return cudaErrorInvalidValue;
}

}  // namespace ppgpu
