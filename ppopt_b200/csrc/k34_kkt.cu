// K3 + K4 - KKT solve by Schur complement / Cholesky and the theta-space optimality + full-dimension test.
// One warp per feasible candidate.
//
// Reference work replaced, per candidate:
//   check_optimality       /root/reference/src/ppopt/mpqp_program.py:203-322   (an (n+t+m+1)-variable LP "max t")
//   optimal_control_law    /root/reference/src/ppopt/mpqp_program.py:146-198   (two LU solves of the KKT matrix)
//   region rows + filters  /root/reference/src/ppopt/utils/mpqp_utils.py:111-126
//   is_full_dimensional    /root/reference/src/ppopt/utils/mpqp_utils.py:323-344 -> chebyshev_ball.py:10-63
// For a nonsingular KKT system x(theta), lambda(theta) are unique affine maps, so the big optimality LP is feasible
// iff the polytope { lambda_act(theta) >= 0, inactive slacks(theta) >= 0, A_t theta <= b_t } is non-empty
// (the same reduction the reference itself uses in mp_solvers/mpqp_combi_graph.py:48-66); its Chebyshev radius then
// decides full dimensionality.  With G = At Qr^-1 At' and V precomputed (host_math.hpp):
//   S = G[act,act] (gather, k'xk')   Lambda = -S^-1 V[act]        (Cholesky + 2 triangular solves, t+1 rhs)
//   lambda rows:   -Lambda_theta[j] . theta <= Lambda_const[j]
//   inactive rows: -(V_theta[i] + G[i,act] Lambda_theta) . theta <= V_const[i] + G[i,act] Lambda_const
// Zero rows (all |a| <= 1e-8) are dropped unless their rhs < -1e-7 (then the candidate is not optimal), rows are
// L2-normalised and  max r : a.theta + r <= f  is solved by the register simplex of lp_core.cuh.
// This kernel is a SCREEN (radius >= PPG_RADIUS_SCREEN); K5 repeats the test on LU-accurate rows before emitting.
#include "common.cuh"
#include "launch.h"
#include "lp_core.cuh"

namespace ppgpu {


// K3p - one THREAD per feasible candidate (small k'): Schur system + multiplier-sign test entirely in registers.
// The warp-per-candidate kernel below spent 85 % of its instructions here with ~11 of 32 lanes active; this stage has
// no cross-lane work at all, so 32 candidates share one instruction stream.  Survivors get PPG_ST_PRE and are the
// only ones k34_kernel still builds rows / runs the Chebyshev LP for.
template <int KC>
__global__ void __launch_bounds__(128)
k3_prefilter_kernel(DevProgram P, const uint64_t* __restrict__ masks, long long n, int k, uint8_t* __restrict__ status) {
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= n) return;
    const uint8_t st = status[idx];
    if (!(st & PPG_ST_FEAS)) return;
    const int t = P.t, t1 = P.t + 1, mi = P.mi, W = P.W;
    const uint64_t* mk = masks + idx * W;
    int act[KC];
#pragma unroll
    for (int a = 0; a < KC; ++a) act[a] = (a < k) ? mask_nth(mk, W, a) : 0;
    double L[KC][KC];
#pragma unroll
    for (int a = 0; a < KC; ++a)
#pragma unroll
        for (int b = 0; b <= a; ++b) L[a][b] = (a < k && b < k) ? __ldg(P.G + (size_t)act[a] * mi + act[b]) : (a == b ? 1.0 : 0.0);
    bool pd = true;
    double Linv[KC];   // 1 / L[j][j]: the 2 (t+1) KC substitutions below multiply instead of dividing (an fp64 division is ~25
                       // instructions; they were a third of this kernel)
#pragma unroll
    for (int j = 0; j < KC; ++j) {
        double d = L[j][j];
#pragma unroll
        for (int c = 0; c < j; ++c) d = fma(-L[j][c], L[j][c], d);
        if (!(d > 0.0)) pd = false;
        const double sd = sqrt(d > 0.0 ? d : 1.0), isd = 1.0 / sd;
        L[j][j] = sd;
        Linv[j] = isd;
#pragma unroll
        for (int i = j + 1; i < KC; ++i) {
            double s2 = L[i][j];
#pragma unroll
            for (int c = 0; c < j; ++c) s2 = fma(-L[i][c], L[j][c], s2);
            L[i][j] = s2 * isd;
        }
    }
    if (!pd) { status[idx] = st | PPG_ST_PRE; return; }  // let the warp kernel report the numeric failure
    bool reject = false;
    // one right-hand side (column of V) at a time keeps the register footprint at KC doubles
    double ub[KC], mx[KC], mag[KC], cst[KC];
#pragma unroll
    for (int a = 0; a < KC; ++a) { ub[a] = 0.0; mx[a] = 0.0; mag[a] = 0.0; cst[a] = 0.0; }
    for (int c = 0; c < t1; ++c) {
        double x[KC];
#pragma unroll
        for (int i = 0; i < KC; ++i) {
            double s2 = (i < k) ? -__ldg(P.V + (size_t)act[i] * t1 + c) : 0.0;
#pragma unroll
            for (int j = 0; j < i; ++j) s2 = fma(-L[i][j], x[j], s2);
            x[i] = s2 * Linv[i];
        }
#pragma unroll
        for (int i = KC - 1; i >= 0; --i) {
            double s2 = x[i];
#pragma unroll
            for (int j = i + 1; j < KC; ++j) s2 = fma(-L[j][i], x[j], s2);
            x[i] = s2 * Linv[i];
        }
        if (c == 0) {
#pragma unroll
            for (int a = 0; a < KC; ++a) { ub[a] = x[a]; mag[a] = fabs(x[a]); cst[a] = x[a]; }
        } else {
            const double lo = __ldg(P.th_lo + c - 1), hi = __ldg(P.th_hi + c - 1);
#pragma unroll
            for (int a = 0; a < KC; ++a) {
                const double av = x[a];
                mx[a] = fmax(mx[a], fabs(av));
                if (av != 0.0) { const double term = fmax(av * lo, av * hi); ub[a] += term; mag[a] += fabs(term); }
            }
        }
    }
#pragma unroll
    for (int a = 0; a < KC; ++a)
        if (a < k) {
            if (mx[a] > PPG_ZERO_ROW) { if (ub[a] < -1e-9 * fmax(1.0, mag[a])) reject = true; }
            // a multiplier that does not depend on theta and is negative: the zero-row rule of the row build (numerically zero
            // row with rhs < -1e-7 => not optimal, mpqp_utils.py:123-125 + the LP) applied before any row is built - 8 % of the
            // level at the 100 x 30 x 6 program (active sets made of box rows only)
            else if (mx[a] <= PPG_ZERO_ROW && cst[a] < -PPG_FEAS_TOL) reject = true;
        }
    (void)t;
    if (!reject) status[idx] = st | PPG_ST_PRE;
}

template <int KC>
static cudaError_t launch_k3p_t(const DevProgram& P, const uint64_t* masks, long long n, int k_act, uint8_t* status, cudaStream_t st) {
    k3_prefilter_kernel<KC><<<(unsigned)((n + 127) / 128), 128, 0, st>>>(P, masks, n, k_act, status);
    return cudaGetLastError();
}

// returns true (and launches) when the thread-per-candidate prefilter covers this level
static bool launch_k3p(const DevProgram& P, const uint64_t* masks, long long n, int k_act, uint8_t* status, cudaStream_t st,
                       cudaError_t* err) {
    *err = cudaSuccess;
    if (k_act < 1 || k_act > 8) return false;
    if (k_act <= 2) *err = launch_k3p_t<2>(P, masks, n, k_act, status, st);
    else if (k_act <= 4) *err = launch_k3p_t<4>(P, masks, n, k_act, status, st);
    else if (k_act <= 6) *err = launch_k3p_t<6>(P, masks, n, k_act, status, st);
    else *err = launch_k3p_t<8>(P, masks, n, k_act, status, st);
    return true;
}

template <int RPT, int DC, int WPC>
__global__ void __launch_bounds__(32 * WPC)
k34_kernel(DevProgram P, const uint64_t* __restrict__ masks, long long n, int k_act, uint8_t* __restrict__ status,
           unsigned long long* __restrict__ queue, unsigned long long* __restrict__ counters, int use_pre, int scan_pt) {
    typedef LpCore<1, RPT, DC> Core;
    extern __shared__ double dyn_smem[];
    __shared__ typename Core::Shared sh_all[WPC];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    typename Core::Shared& sh = sh_all[warp];
    const int t = P.t, t1 = P.t + 1, mi = P.mi, W = P.W, kmax = k_act;
    // per-warp scratch: S (kmax x kmax), Lam (kmax x t1), act (kmax ints)
    const size_t per_warp = (size_t)kmax * kmax + (size_t)kmax * t1 + (size_t)((kmax + 1) / 2 + 1);
    double* S = dyn_smem + per_warp * warp;
    double* Lam = S + (size_t)kmax * kmax;
    int* act = reinterpret_cast<int*>(Lam + (size_t)kmax * t1);
    unsigned long long n_lp = 0, n_piv = 0, n_work = 0, n_num = 0;
    // the level is scanned in blocks of 32 * scan_pt status bytes per queue item (the prefilter leaves a few per cent of
    // the candidates: one atomic and one dependent status load per candidate would dominate)
    const int blk = 32 * scan_pt;
    const long long nblocks = (n + blk - 1) / blk;
    for (;;) {
        unsigned long long v = 0;
        if (lane == 0) v = atomicAdd(queue, 1ull);
        const long long item = (long long)__shfl_sync(PPG_FULL, v, 0);
        if (item >= nblocks) break;
        const long long c0 = item * blk + (long long)lane * scan_pt;
        unsigned need = 0;   // bit j: candidate c0 + j is feasible and passed the prefilter
        {
            uint8_t sb[16];
            if (scan_pt == 16 && c0 + 16 <= n && (reinterpret_cast<uintptr_t>(status + c0) & 15) == 0) {
                const uint4 q = *reinterpret_cast<const uint4*>(status + c0);
                const unsigned w4[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
                for (int j = 0; j < 16; ++j) sb[j] = (uint8_t)(w4[j >> 2] >> ((j & 3) * 8));
            } else {
#pragma unroll
                for (int j = 0; j < 16; ++j) sb[j] = (j < scan_pt && c0 + j < n) ? status[c0 + j] : 0;
            }
#pragma unroll
            for (int j = 0; j < 16; ++j)
                if ((sb[j] & PPG_ST_FEAS) && (!use_pre || (sb[j] & PPG_ST_PRE))) need |= 1u << j;
        }
        for (;;) {
        const unsigned bal = __ballot_sync(PPG_FULL, need != 0);
        if (!bal) break;
        const int src = __ffs((int)bal) - 1;
        const unsigned nm = __shfl_sync(PPG_FULL, need, src);
        const int jb = __ffs((int)nm) - 1;
        if (lane == src) need &= need - 1;
        const long long idx = item * blk + (long long)src * scan_pt + jb;
        uint8_t st = status[idx];
        if (use_pre) st &= (uint8_t)~PPG_ST_PRE;
        const uint64_t* mk = masks + idx * W;
        const int k = kmax;
        __syncwarp();
        for (int j = lane; j < k; j += 32) act[j] = mask_nth(mk, W, j);
        __syncwarp();
        for (int e = lane; e < k * k; e += 32) {
            const int a = e / k, b2 = e - a * k;
            S[e] = __ldg(P.G + (size_t)act[a] * mi + act[b2]);
        }
        __syncwarp();
        // Cholesky (lower), right-looking, lanes over rows
        bool pd = true;
        for (int j = 0; j < k; ++j) {
            const double d = S[j * k + j];
            if (!(d > 0.0)) { pd = false; break; }
            const double sd = sqrt(d);
            __syncwarp();
            for (int i = j + 1 + lane; i < k; i += 32) S[i * k + j] /= sd;
            if (lane == 0) S[j * k + j] = sd;
            __syncwarp();
            for (int i = j + 1 + lane; i < k; i += 32) {
                const double lij = S[i * k + j];
                for (int c = j + 1; c <= i; ++c) S[i * k + c] = fma(-lij, S[c * k + j], S[i * k + c]);
            }
            __syncwarp();
        }
        bool pass = false;
        bool numeric = false, thin = false;
        if (!pd) {
            numeric = true;
        } else {
            // Lambda = -S^-1 V[act]; lane c handles rhs column c (0 = constant term)
            if (lane < t1) {
                for (int i = 0; i < k; ++i) {
                    double s = -__ldg(P.V + (size_t)act[i] * t1 + lane);
                    for (int j = 0; j < i; ++j) s = fma(-S[i * k + j], Lam[j * t1 + lane], s);
                    Lam[i * t1 + lane] = s / S[i * k + i];
                }
                for (int i = k - 1; i >= 0; --i) {
                    double s = Lam[i * t1 + lane];
                    for (int j = i + 1; j < k; ++j) s = fma(-S[j * k + i], Lam[j * t1 + lane], s);
                    Lam[i * t1 + lane] = s / S[i * k + i];
                }
            }
            __syncwarp();
            // cheap NECESSARY condition before the expensive part: every nonzero multiplier row must be able to reach
            // lambda_j(theta) > 0 somewhere in the bounding box of Theta (else the theta-polytope is empty)
            bool reject = false;
            for (int j = lane; j < k; j += 32) {
                double ub = Lam[j * t1], mx = 0.0, mag = fabs(Lam[j * t1]);
                for (int c = 0; c < t; ++c) {
                    const double a = Lam[j * t1 + 1 + c];
                    const double lo = __ldg(P.th_lo + c), hi = __ldg(P.th_hi + c);
                    mx = fmax(mx, fabs(a));
                    if (a != 0.0) { const double term = fmax(a * lo, a * hi); ub += term; mag += fabs(term); }
                }
                if (mx > PPG_ZERO_ROW) { if (ub < -1e-9 * fmax(1.0, mag)) reject = true; }
                else if (mx <= PPG_ZERO_ROW && Lam[j * t1] < -PPG_FEAS_TOL) reject = true;   // zero-row rule, see k3_prefilter_kernel
            }
            if (__any_sync(PPG_FULL, reject)) {
                if (use_pre && lane == 0) status[idx] = st;
                continue;  // not optimal: status keeps PPG_ST_FEAS only
            }
            // region rows straight into the tableau registers: T[.][0] = f, T[.][1..t] = a, T[.][t+1] = 1 (the s column)
            double T[RPT][DC];
            int rflag[RPT];
            bool zero_viol = false;
            static_for<RPT>([&](auto RR) {
                constexpr int rr = decltype(RR)::value;
                const int row = rr * 32 + lane;
#pragma unroll
                for (int c = 0; c < DC; ++c) T[rr][c] = 0.0;
                rflag[rr] = 0;
                if (row < P.R0) {
                    if (row < mi) {
                        if (mask_test(mk, row)) {
                            const int pos = mask_rank(mk, row);
#pragma unroll
                            for (int c = 0; c < DC; ++c)
                                if (c < t1) T[rr][c] = (c == 0) ? Lam[pos * t1] : -Lam[pos * t1 + c];
                        } else {
#pragma unroll
                            for (int c = 0; c < DC; ++c)
                                if (c < t1) T[rr][c] = __ldg(P.V + (size_t)row * t1 + c);
                            for (int a = 0; a < k; ++a) {
                                const double g = __ldg(P.G + (size_t)row * mi + act[a]);
#pragma unroll
                                for (int c = 0; c < DC; ++c)
                                    if (c < t1) T[rr][c] = fma(g, Lam[a * t1 + c], T[rr][c]);
                            }
#pragma unroll
                            for (int c = 1; c < DC; ++c)
                                if (c < t1) T[rr][c] = -T[rr][c];
                        }
                    } else {
                        const int o = row - mi;
                        T[rr][0] = __ldg(P.b_t + o);
#pragma unroll
                        for (int c = 1; c < DC; ++c)
                            if (c < t1) T[rr][c] = __ldg(P.A_t + (size_t)o * t + c - 1);
                    }
                    double mx = 0.0, nn = 0.0;
#pragma unroll
                    for (int c = 1; c < DC; ++c)
                        if (c < t1) { mx = fmax(mx, fabs(T[rr][c])); nn = fma(T[rr][c], T[rr][c], nn); }
                    if (!(mx <= PPG_ZERO_ROW)) {
                        const double inv = 1.0 / sqrt(nn);
#pragma unroll
                        for (int c = 0; c < DC; ++c)
                            if (c < t1) T[rr][c] *= inv;
                        rflag[rr] = 1;
                    } else if (T[rr][0] < -PPG_FEAS_TOL) {
                        zero_viol = true;
                    }
                }
            });
            const bool any_viol = __any_sync(PPG_FULL, zero_viol);
            if (!any_viol) {
                if (t == 1) {
                    // interval [lo, hi] of the 1-D polytope (get_bounds_1d, mpqp_utils.py:304-315)
                    double lo = -CUDART_INF, hi = CUDART_INF;
                    static_for<RPT>([&](auto RR) {
                        constexpr int rr = decltype(RR)::value;
                        if (rflag[rr] == 1) {
                            const double q = T[rr][0] / T[rr][1];
                            if (T[rr][1] > 0.0) hi = fmin(hi, q); else lo = fmax(lo, q);
                        }
                    });
#pragma unroll
                    for (int o = 16; o > 0; o >>= 1) {
                        lo = fmax(lo, shfl_xor_d(lo, o));
                        hi = fmin(hi, shfl_xor_d(hi, o));
                    }
                    pass = (lo + 0.5 * PPG_WIDTH_1D <= hi);
                } else {
                    static_for<RPT>([&](auto RR) {
                        constexpr int rr = decltype(RR)::value;
                        if (rflag[rr] == 1) {
#pragma unroll
                            for (int c = 0; c < DC; ++c)
                                if (c == t1) T[rr][c] = 1.0;
                        }
                    });
                    LpOut res = Core::solve(sh, T, rflag, P.R0, t1, PPG_RADIUS_SCREEN, false, lane);
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

template <int RPT, int DC>
static cudaError_t launch_k34_t(const DevProgram& P, const uint64_t* masks, long long n, int k_act, uint8_t* status,
                                unsigned long long* queue, unsigned long long* counters, int sm_count, cudaStream_t st, int use_pre) {
    constexpr int WPC = 4;
    auto kern = k34_kernel<RPT, DC, WPC>;
    const size_t per_warp = (size_t)k_act * k_act + (size_t)k_act * (P.t + 1) + (size_t)((k_act + 1) / 2 + 1);
    const size_t smem = per_warp * WPC * sizeof(double);
    cudaError_t e;
    if ((e = fit_smem(kern, smem)) != cudaSuccess) return e;
    int occ = 0;
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, 32 * WPC, smem);
    if (e != cudaSuccess) return e;
    if (occ < 1) occ = 1;
    long long grid = (long long)sm_count * occ;
    const long long need = (n + WPC - 1) / WPC;
    if (grid > need) grid = need;
    if (grid < 1) grid = 1;
    // one status byte per lane and queue item: 32x fewer atomics than one item per candidate, and still ~1 LP per item
    // (16 bytes per lane measured slower: the survivors cluster and a warp then owns dozens of 100 us LPs in a row)
    const int scan_pt = 1;
    kern<<<(unsigned)grid, 32 * WPC, smem, st>>>(P, masks, n, k_act, status, queue, counters, use_pre, scan_pt);
    return cudaGetLastError();
}

#define K34_RPT_SWITCH(DCV)                                                                                  \
    if (P.R0 <= 32) return launch_k34_t<1, DCV>(P, masks, n, k_act, status, queue, counters, sm_count, st, use_pre);  \
    if (P.R0 <= 64) return launch_k34_t<2, DCV>(P, masks, n, k_act, status, queue, counters, sm_count, st, use_pre);  \
    if (P.R0 <= 128) return launch_k34_t<4, DCV>(P, masks, n, k_act, status, queue, counters, sm_count, st, use_pre); \
    if (P.R0 <= 256) return launch_k34_t<8, DCV>(P, masks, n, k_act, status, queue, counters, sm_count, st, use_pre); \
    return cudaErrorInvalidValue;

cudaError_t launch_k34(const DevProgram& P, const uint64_t* masks, long long n, int k_act, uint8_t* status,
                       unsigned long long* queue, unsigned long long* counters, int sm_count, cudaStream_t st) {
    cudaError_t perr;
    const int use_pre = launch_k3p(P, masks, n, k_act, status, st, &perr) ? 1 : 0;
    if (perr != cudaSuccess) return perr;
    {
        // production path: the compact shared-memory form (k34c_compact.cu); the register form below is kept for programs
        // whose tableau does not fit shared memory and as the A/B reference (PPGPU_K34_COMPACT=0)
        bool handled = false;
        const cudaError_t e = launch_k34_compact(P, masks, n, k_act, status, queue, counters, sm_count, st, use_pre, &handled);
        if (e != cudaSuccess || handled) return e;
    }
    if (P.t + 2 <= 8) { K34_RPT_SWITCH(8) }
    if (P.t + 2 <= 16) { K34_RPT_SWITCH(16) }
    return cudaErrorInvalidValue;
}

// general (non-Gram) path: every feasible candidate the reference would pass to check_optimality is handed to K5.
// mpLP: only |active set| == n can be optimal (mplp_program.py:472-473).
__global__ void mark_general_kernel(long long n, int pass_all, uint8_t* __restrict__ status) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) {
        const uint8_t st = status[i];
        if ((st & PPG_ST_FEAS) && pass_all) status[i] = st | PPG_ST_OPT;
    }
}

cudaError_t launch_mark_general(const DevProgram& P, long long n, int k_act, uint8_t* status, cudaStream_t st) {
    const int pass_all = P.is_qp ? 1 : ((P.ne + k_act == P.n) ? 1 : 0);
    if (n <= 0) return cudaSuccess;
    mark_general_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(n, pass_all, status);
    return cudaGetLastError();
}

}  // namespace ppgpu
