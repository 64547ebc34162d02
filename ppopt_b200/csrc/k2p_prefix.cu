// K2a, prefix form - feasibility CERTIFICATES by projected relaxation with the Gram matrix projected ONCE PER PREFIX.
//
// Same question and same method as k2a_relax.cu (check_feasibility, /root/reference/src/ppopt/mplp_program.py:411-444;
// Agmon-Motzkin relaxation inside the affine subspace of the active rows, exact verification of the final point, never
// decides infeasibility), restructured around how an enumeration level is laid out: the level is in lexicographic order
// (mpqp_combinatorial.py:60-61 extends parent by parent), so candidates that share their first k'-2 active rows - the
// PREFIX - are contiguous, ~460 of them on average at level 5 of the 100x30x6 program.  For a prefix P
//     n_j = g_j - G_P' W[:,j],  W = (Gam[P,P])^-1 Gam[P,:]          (generators of the null space of G_P)
//     Gp[j][r] = g_r . n_j = Gam[j][r] - sum_a Gam[P_a][r] W[a][j]   (R0 x R0, shared memory, built once per prefix)
// and a candidate P + {a, b} only has to deflate its own two rows:
//     step along row j:  v_r -= tau ( Gp[j][r] - m0 Gp[a][r] - m1 Gp[b][r] ),   (m0 m1) = (Gp[j][a] Gp[j][b]) S2^-1
// i.e. 3 FMAs per row and step instead of 1 + k', no per-candidate factorisation, and every operand comes from shared
// memory.  A sub-warp GROUP of LANES lanes owns a candidate (16 lanes x 7 rows or 8 lanes x 14 rows for 112 rows), so one
// instruction stream carries 2 or 4 candidates and the per-step bookkeeping (arg-max key, stall detector, step length)
// is paid once for all of them.  The groups run independent candidates and refill themselves from the CTA's segment
// counter; only set-up and verification are executed group by group.
//
// The point is carried as its coefficient vector over the generators (coef[j] in shared memory, one RMW per step);
// on convergence EVERY row - prefix and suffix equalities included - is re-evaluated from the coefficients:
//     s_r = v0_r + sum_j coef_j Gp[j][r] + x_a Gp[a][r] + x_b Gp[b][r],   v0 = residuals of the min-norm point of P
// Gp[j][r] is, up to the rounding of its own evaluation, the exact inner product of g_r with the concrete vector n_j
// defined by the NUMERIC W, so this is an honest evaluation of a concrete point (same error model as k2a_relax.cu's
// Gram-space verification), not a statement that relies on W being exact.
// Candidates that cannot be certified leave the exact residuals of their last iterate for K2 (DevProgram::warm_*).
#include "common.cuh"
#include "launch.h"
#include "lp_core.cuh"

#include <cstdlib>

namespace ppgpu {

constexpr int K2P_CHUNK = 1024;   // candidates a CTA stages per work item
constexpr int K2P_PMAX = 16;      // longest prefix (k' - 2) this kernel handles
constexpr double K2P_OMEGA = 1.35, K2P_OMEGA2 = 1.8;   // see k2a_relax.cu (scanned on the 100x30x6 program)
constexpr int K2P_STALL1 = 16, K2P_STALL2 = 48;
constexpr unsigned K2P_TODO = 1u << 16;

struct K2pCtl { long long base; unsigned long long pf[4]; unsigned long long n_try, n_ok, n_it; int next; int seg_end; int any; int valid; };

__device__ __forceinline__ double k2p_lds(unsigned a) {
    double x;
    asm volatile("ld.shared.f64 %0, [%1];" : "=d"(x) : "r"(a));
    return x;
}
__device__ __forceinline__ void k2p_sts(unsigned a, double x) { asm volatile("st.shared.f64 [%0], %1;" ::"r"(a), "d"(x) : "memory"); }
__device__ __forceinline__ unsigned k2p_ldsu(unsigned a) {
    unsigned x;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(x) : "r"(a));
    return x;
}

// words of candidate i with its suffix rows (bits a and b) cleared = the prefix
__device__ __forceinline__ void k2p_prefix_words(const uint64_t* m, int W, unsigned ab, uint64_t (&out)[4]) {
    const int a = ab & 255, b = (ab >> 8) & 255;
#pragma unroll
    for (int w = 0; w < 4; ++w) {
        uint64_t x = w < W ? m[w] : 0ull;
        if ((a >> 6) == w) x &= ~(1ull << (a & 63));
        if ((b >> 6) == w) x &= ~(1ull << (b & 63));
        out[w] = x;
    }
}
// index of the j-th (0-based) set bit of a 4-word mask held in registers
__device__ __forceinline__ int k2p_nth(const uint64_t (&m)[4], int j) {
    int r = -1;
    bool done = false;
#pragma unroll
    for (int w = 0; w < 4; ++w) {
        const int c = __popcll(m[w]);
        if (!done && j < c) {
            const unsigned lo = (unsigned)m[w], hi = (unsigned)(m[w] >> 32);
            const int cl = __popc(lo);
            r = j < cl ? w * 64 + (int)__fns(lo, 0, j + 1) : w * 64 + 32 + (int)__fns(hi, 0, j - cl + 1);
            done = true;
        }
        if (!done) j -= c;
    }
    return r;
}

// max of `key` over each group of LANES lanes, on every lane of the group: one redux.sync per group (the whole warp takes
// part, lanes of the other groups contribute INT_MIN) - a 4-step shuffle ladder is ~110 cycles of dependent latency, 32 / LANES
// independent redux instructions ~30
template <int LANES>
__device__ __forceinline__ int k2p_group_max(int key, int g) {
    if constexpr (LANES == 32) {
        return __reduce_max_sync(PPG_FULL, key);
    } else {
        int out = 0;
#pragma unroll
        for (int q = 0; q < 32 / LANES; ++q) {
            const int m = __reduce_max_sync(PPG_FULL, g == q ? key : (int)0x80000000);
            if (g == q) out = m;
        }
        return out;
    }
}

template <int LANES, int RL, int THREADS>
__global__ void __launch_bounds__(THREADS, 1)
k2p_relax_kernel(DevProgram P, const uint64_t* __restrict__ masks, long long n, int k_act, uint8_t* __restrict__ status,
                 unsigned long long* __restrict__ queue, unsigned long long* __restrict__ counters, int max_iter,
                 int max_iter2, int chunk, int scratch_doubles) {
    constexpr int LD = RL * LANES;
    constexpr int NG = 32 / LANES;
    constexpr unsigned ROWB = LD * 8;       // bytes per row of Gp
    constexpr unsigned SLOTB = LANES * 8;   // bytes between a lane's consecutive rows
    extern __shared__ double sm[];
    const int R0 = P.R0, W = P.W, dc0 = P.dc0;
    double* Gp = sm;                       // R0 x LD
    double* v0 = Gp + (size_t)R0 * LD;     // LD
    double* scr = v0 + LD;                 // build scratch / per-group coefficient vectors
    uint64_t* cmask = reinterpret_cast<uint64_t*>(scr + scratch_doubles);   // chunk x W
    unsigned* cab = reinterpret_cast<unsigned*>(cmask + (size_t)K2P_CHUNK * W);   // chunk: a | b << 8 | todo << 16 | status << 24
    double* scr_v = reinterpret_cast<double*>(cab + K2P_CHUNK);   // per warp: exact residuals on their way back to a group
    __shared__ K2pCtl ctl;
    __shared__ int pr_s[K2P_PMAX];
    __shared__ double w0_s[K2P_PMAX];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane / LANES, gl = lane % LANES;
    const unsigned gmask = (LANES == 32 ? 0xffffffffu : ((1u << LANES) - 1u)) << (LANES * g);
    const int gsrc = LANES * g;
    const int p = k_act >= 2 ? k_act - 2 : 0;
    const bool has_b = k_act >= 2;
    const double* __restrict__ Gam = P.Gam;
    const double* __restrict__ T0 = P.T0;
    const int ktol = (__double2hiint(PPG_FEAS_TOL * 0.999) & ~127) | 127;
    // 32-bit shared addresses (opaque to the compiler so that they stay in registers)
    unsigned gp_sa = (unsigned)__cvta_generic_to_shared(Gp);
    unsigned v0_sa = (unsigned)__cvta_generic_to_shared(v0);
    unsigned coef_sa = (unsigned)__cvta_generic_to_shared(scr + (size_t)(warp * NG + g) * LD);
    unsigned cab_sa = (unsigned)__cvta_generic_to_shared(cab);
    asm volatile("" : "+r"(gp_sa), "+r"(v0_sa), "+r"(coef_sa), "+r"(cab_sa));
    const unsigned lane_off = (unsigned)gl * 8u;
    int kid[RL];
#pragma unroll
    for (int rr = 0; rr < RL; ++rr) { kid[rr] = rr * LANES + gl; asm volatile("" : "+r"(kid[rr])); }
    if (tid == 0) { ctl.n_try = 0ull; ctl.n_ok = 0ull; ctl.n_it = 0ull; }

    for (;;) {
        __syncthreads();   // everybody is done with the previous chunk (ctl, cmask, cab)
        if (tid == 0) ctl.base = (long long)atomicAdd(queue, (unsigned long long)chunk);
        __syncthreads();
        const long long base = ctl.base;
        if (base >= n) break;
        const int cn = (int)((n - base) < (long long)chunk ? (n - base) : (long long)chunk);
        // whether a candidate needs work; PPG_ST_PRE: the vertex walk proved it infeasible (k2w_walk.cu).  A chunk with
        // nothing to do is left before its masks are read and its prefixes projected - after a walked level that is
        // nearly every chunk.  (No candidate's result depends on the chunk around it: a prefix cut by a chunk boundary is
        // simply projected twice, and chunk sizes already vary with n.)
        int any_chunk = 0;
        for (int i = tid; i < cn; i += THREADS) {
            const uint8_t sb = status[base + i];
            const bool todo = (sb & PPG_ST_RANK) && !(sb & (PPG_ST_FEAS | PPG_ST_PRE));
            cab[i] = (todo ? K2P_TODO : 0u) | ((unsigned)sb << 24);
            any_chunk |= todo;
        }
        if (!__syncthreads_or(any_chunk)) continue;
        for (int i = tid; i < cn; i += THREADS) {
            // stage the candidate: mask words, its two highest rows (the suffix)
            int hi1 = 0, hi2 = 0;
            for (int w = 0; w < W; ++w) {
                const uint64_t x = masks[(base + i) * W + w];
                cmask[(size_t)i * W + w] = x;
                if (x) {
                    const int t1 = w * 64 + 63 - __clzll((long long)x);
                    const uint64_t y = x & ~(1ull << (t1 & 63));
                    hi2 = y ? w * 64 + 63 - __clzll((long long)y) : hi1;
                    hi1 = t1;
                }
            }
            const unsigned a = has_b ? (unsigned)hi2 : (unsigned)hi1, b = (unsigned)hi1;
            cab[i] |= a | (b << 8);
        }
        __syncthreads();
        int s0 = 0;
        while (s0 < cn) {
            // ---- segment [s0, s1): candidates with the prefix of candidate s0
            uint64_t pf0[4];
            k2p_prefix_words(cmask + (size_t)s0 * W, W, k_act >= 1 ? cab[s0] : 0xffffu, pf0);
            if (tid == 0) { ctl.seg_end = cn; ctl.any = 0; ctl.valid = 1; ctl.pf[0] = pf0[0]; ctl.pf[1] = pf0[1]; ctl.pf[2] = pf0[2]; ctl.pf[3] = pf0[3]; }
            __syncthreads();
            for (int i = s0 + 1 + tid; i < cn; i += THREADS) {
                uint64_t pf[4];
                k2p_prefix_words(cmask + (size_t)i * W, W, cab[i], pf);
                const bool same = pf[0] == pf0[0] && pf[1] == pf0[1] && pf[2] == pf0[2] && pf[3] == pf0[3];
                if (!same) { atomicMin(&ctl.seg_end, i); break; }   // sorted level: later ones differ as well
            }
            __syncthreads();
            const int s1 = ctl.seg_end;
            for (int i = s0 + tid; i < s1; i += THREADS)
                if (cab[i] & K2P_TODO) atomicOr(&ctl.any, 1);
            __syncthreads();
            const int any_todo = ctl.any;
            if (!any_todo) { s0 = s1; __syncthreads(); continue; }   // (ctl is rewritten at the top of the loop)

            // ---- build Gp and v0 for this prefix
            double* PR = scr;                       // p x LD   rows Gam[P_a][:]
            double* Wt = scr + (size_t)p * LD;      // p x LD   W[a][j]
            double* Sp = Wt + (size_t)p * LD;       // p x p    LDL' of Gam[P,P] (unit lower L below the diagonal, d on it)
            if (tid < p) pr_s[tid] = k2p_nth(pf0, tid);
            __syncthreads();
            for (int e = tid; e < p * LD; e += THREADS) {
                const int a = e / LD, r = e - a * LD;
                const double x = r < R0 ? __ldg(Gam + (size_t)pr_s[a] * R0 + r) : 0.0;
                PR[e] = x;
                Wt[e] = x;
            }
            for (int e = tid; e < p * p; e += THREADS) Sp[e] = __ldg(Gam + (size_t)pr_s[e / p] * R0 + pr_s[e % p]);
            if (tid < p) w0_s[tid] = __ldg(T0 + (size_t)pr_s[tid] * dc0);
            __syncthreads();
            if (warp == 0 && p > 0) {
                // right-looking LDL' (p <= 16): column j, then the trailing update, lanes over rows
                for (int j = 0; j < p; ++j) {
                    const double d = Sp[j * p + j];
                    if (!(d > 1e-12)) { if (lane == 0) ctl.valid = 0; break; }
                    const double dinv = 1.0 / d;
                    __syncwarp();
                    double lij = 0.0;
                    if (lane > j && lane < p) lij = Sp[lane * p + j] * dinv;
                    __syncwarp();
                    if (lane > j && lane < p) {
                        for (int c = j + 1; c <= lane; ++c) Sp[lane * p + c] = fma(-lij, Sp[c * p + j], Sp[lane * p + c]);
                    }
                    __syncwarp();
                    if (lane > j && lane < p) Sp[lane * p + j] = lij;
                    __syncwarp();
                }
            }
            __syncthreads();
            const bool valid = ctl.valid != 0;
            if (valid && p > 0) {
                // W[:, j] = S^-1 Gam[P, j] (thread per column), w0 = S^-1 h_P (one more thread)
                if (tid < R0) {
                    for (int i = 1; i < p; ++i) {
                        double x = Wt[i * LD + tid];
                        for (int c = 0; c < i; ++c) x = fma(-Sp[i * p + c], Wt[c * LD + tid], x);
                        Wt[i * LD + tid] = x;
                    }
                    for (int i = 0; i < p; ++i) Wt[i * LD + tid] /= Sp[i * p + i];
                    for (int i = p - 2; i >= 0; --i) {
                        double x = Wt[i * LD + tid];
                        for (int c = i + 1; c < p; ++c) x = fma(-Sp[c * p + i], Wt[c * LD + tid], x);
                        Wt[i * LD + tid] = x;
                    }
                } else if (tid == THREADS - 1) {
                    for (int i = 1; i < p; ++i) {
                        double x = w0_s[i];
                        for (int c = 0; c < i; ++c) x = fma(-Sp[i * p + c], w0_s[c], x);
                        w0_s[i] = x;
                    }
                    for (int i = 0; i < p; ++i) w0_s[i] /= Sp[i * p + i];
                    for (int i = p - 2; i >= 0; --i) {
                        double x = w0_s[i];
                        for (int c = i + 1; c < p; ++c) x = fma(-Sp[c * p + i], w0_s[c], x);
                        w0_s[i] = x;
                    }
                }
            }
            __syncthreads();
            if (valid) {
                for (int e = tid; e < R0 * LD; e += THREADS) {
                    const int j = e / LD, r = e - j * LD;
                    double x = 0.0;
                    if (r < R0) {
                        x = __ldg(Gam + (size_t)j * R0 + r);
                        for (int a = 0; a < p; ++a) x = fma(-PR[a * LD + r], Wt[a * LD + j], x);
                    }
                    Gp[e] = x;
                }
                if (tid < LD) {
                    double x = 0.0;
                    if (tid < R0) {
                        x = -__ldg(T0 + (size_t)tid * dc0);
                        for (int a = 0; a < p; ++a) x = fma(PR[a * LD + tid], w0_s[a], x);
                    }
                    v0[tid] = x;
                }
            }
            if (tid == 0) ctl.next = s0;
            __syncthreads();   // Gp / v0 complete, scratch free for the coefficient vectors

            // ---- candidates of the segment: every group pulls one after the other
            if (valid) {
                bool have = false, drained = false;
                int mode = 0;            // 0 stepping, 1 converged (verify), 2 giving up (hand over)
                int ci = 0;              // position of the current candidate in the staged chunk
                unsigned cw = 0;         // its staged word
                unsigned a_off = 0, b_off = 0, park = 0;
                double i11 = 0.0, i12 = 0.0, i22 = 0.0;
                double v[RL], ca[RL], cb[RL];
                int it = 0, it_evt = 0, it_end = 0, next_chk = 0, wref = 0, rechecks = 0, nst = 0;
                bool second = false;
                const bool lead = lane_off == 0u;   // lane 0 of the group
                // which lanes report what in the one vote of an iteration: lane 0 of a group "wants a verification",
                // lane 1 "drained"
                constexpr unsigned LEADS = LANES == 32 ? 1u : (LANES == 16 ? 0x00010001u : 0x01010101u);
                for (;;) {
                    if (!have && !drained) {
                        if (lead) {
                            unsigned w;
                            do {
                                ci = atomicAdd(&ctl.next, 1);
                                w = ci < s1 ? k2p_ldsu(cab_sa + 4u * (unsigned)ci) : 0u;
                            } while (ci < s1 && !(w & K2P_TODO));
                        }
                        ci = __shfl_sync(gmask, ci, gsrc);
                        if (ci >= s1) {
                            drained = true;   // this group is done with the segment (it keeps helping with verifications)
                        } else {
                            // ---- set-up: the candidate's own two rows, start point = min-norm point of its equalities
                            cw = k2p_ldsu(cab_sa + 4u * (unsigned)ci);
                            const unsigned a_row = cw & 255u, b_row = (cw >> 8) & 255u;
                            a_off = a_row * 8u; b_off = b_row * 8u;
                            const unsigned rpa = gp_sa + a_row * ROWB, rpb = gp_sa + b_row * ROWB;
                            const double s11 = k2p_lds(rpa + a_off);
                            const double s12 = has_b ? k2p_lds(rpa + b_off) : 0.0;
                            const double s22 = has_b ? k2p_lds(rpb + b_off) : 1.0;
                            const double det = fma(s11, s22, -s12 * s12);
                            if (lead) atomicAdd(&ctl.n_try, 1ull);
                            if (s11 > 1e-12 && s22 > 1e-12 && det > 1e-12 * s11 * s22) {   // else: left to the simplex
                                double dinv;
                                asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(dinv) : "d"(det));
                                dinv = dinv * fma(-det, dinv, 2.0);
                                dinv = dinv * fma(-det, dinv, 2.0);
                                i11 = s22 * dinv; i12 = -s12 * dinv; i22 = has_b ? s11 * dinv : 0.0;
                                const double va = k2p_lds(v0_sa + a_off), vb = has_b ? k2p_lds(v0_sa + b_off) : 0.0;
                                const double xa = fma(i11, va, i12 * vb), xb = fma(i12, va, i22 * vb);
                                park = 0;
#pragma unroll
                                for (int rr = 0; rr < RL; ++rr) {
                                    const unsigned o = lane_off + rr * SLOTB;
                                    const int r = kid[rr];
                                    ca[rr] = k2p_lds(rpa + o);
                                    cb[rr] = has_b ? k2p_lds(rpb + o) : 0.0;
                                    // parked rows: the prefix (segment-wide), the candidate's own two, the padding beyond R0
                                    const bool pk = r >= R0 || r == (int)a_row || r == (int)b_row ||
                                                    (r < P.mi && ((ctl.pf[(r >> 6) & 3] >> (r & 63)) & 1ull));
                                    park |= (pk ? 1u : 0u) << rr;
                                    const double s = fma(-xb, cb[rr], fma(-xa, ca[rr], k2p_lds(v0_sa + o)));
                                    v[rr] = pk ? -1e300 : s;   // parked: never the maximum
                                    k2p_sts(coef_sa + o, 0.0);
                                }
                                it = 0; it_end = max_iter; next_chk = 0; it_evt = 0; wref = 0; rechecks = 0; nst = 0;
                                second = max_iter2 <= 0;
                                mode = 0;
                                have = true;
                            }
                        }
                    }
                    // ---- the one convergence point of an iteration: the groups vote (and the barrier orders the coefficient
                    // stores of a set-up before the first read-modify-write)
                    __syncwarp();
                    // ---- most violated row of every group: arg-max over keys = high word of the residual with the row index
                    // in its 7 low bits.  Every lane takes part (full-mask shuffles; the ladder never leaves a group), groups
                    // that are not stepping carry a harmless key and their updates below are switched off by tau = 0.
                    const bool stepping = have && mode == 0;
                    int kmax = 0;
#pragma unroll
                    for (int rr = 0; rr < RL; ++rr) kmax = max(kmax, (__double2hiint(v[rr]) & ~127) | kid[rr]);
#pragma unroll
                    for (int o = LANES / 2; o > 0; o >>= 1) kmax = max(kmax, __shfl_xor_sync(PPG_FULL, kmax, o));
                    const int wkey = kmax;
                    bool go = stepping && wkey > ktol;
                    if (stepping) {
                        if (wkey <= ktol) mode = 1;
                        if (go && it >= it_evt) {
                            // stall detector (see k2a_relax.cu): not halving the worst violation in 16 steps -> longer
                            // stride, then the simplex.  Visited every 16 / 48 steps and at the end of a budget.
                            bool stalled = it >= it_end;
                            if (!stalled) {
                                stalled = it != 0 && wkey > wref - 0x100000;
                                wref = wkey;
                                next_chk = it + (second ? K2P_STALL2 : K2P_STALL1);
                            }
                            if (stalled) {
                                if (second) {
                                    mode = 2;
                                    go = false;
                                } else {
                                    second = true;
                                    it_end = it + max_iter2;
                                    wref = wkey;
                                    next_chk = it + K2P_STALL2;
                                }
                            }
                            it_evt = min(it_end, next_chk);
                        }
                        ++it;
                    }
                    {
                        // ---- one relaxation step along row j inside the subspace of the active rows (no branch: a group
                        // that is not stepping runs it with tau = 0 and writes nothing)
                        const unsigned j = stepping ? ((unsigned)wkey & 127u) : 0u;   // (idle groups: a valid row, results unused)
                        const unsigned rowb = gp_sa + j * ROWB;
                        const unsigned rowl = rowb + lane_off;
                        const double ga = k2p_lds(rowb + a_off), gb = k2p_lds(rowb + b_off), gjj = k2p_lds(rowb + j * 8u);
                        const double cold = lead ? k2p_lds(coef_sa + j * 8u) : 0.0;   // (issued early: its latency overlaps the step)
                        const double m0 = fma(ga, i11, gb * i12), m1 = fma(ga, i12, gb * i22);
                        const double nn = fma(-m1, gb, fma(-m0, ga, gjj));   // |N g_j|^2
                        const bool okn = nn > 1e-12;
                        if (go && !okn) mode = 2;   // row j lies in the span of the active rows: leave it to the LP
                        go = go && okn;
                        const double wmax = __hiloint2double(wkey & ~127, 0);   // its violation, rounded down by < 2^-13
                        double rnn;
                        asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(rnn) : "d"(nn));
                        double tau = ((second ? K2P_OMEGA2 : K2P_OMEGA) * wmax) * rnn;
                        tau = go ? tau : 0.0;
                        const double t0 = tau * m0, t1 = tau * m1;
#pragma unroll
                        for (int rr = 0; rr < RL; ++rr) {
                            const double x = k2p_lds(rowl + rr * SLOTB);
                            v[rr] = fma(t1, cb[rr], fma(t0, ca[rr], fma(-tau, x, v[rr])));
                        }
                        if (go && lead) k2p_sts(coef_sa + j * 8u, cold - tau);
                        nst += go ? 1 : 0;
                    }
                    // one vote: lane 0 of every group reports "wants a verification", lane 1 "drained"
                    const unsigned bal = __ballot_sync(PPG_FULL, lead ? (have && mode != 0) : drained);
                    if (((bal >> 1) & LEADS) == LEADS) break;
                    unsigned want = bal & LEADS;
                    // ---- verification / hand-over, one group at a time with the WHOLE warp doing the arithmetic:
                    // exact residuals of the group's current point from its coefficients, all rows (32 lanes x RW rows)
                    while (want) {
                        constexpr int RW = (LD + 31) / 32;
                        __syncwarp();   // lane 0's coefficient read-modify-writes are visible to the whole warp
                        const int og = (__ffs((int)want) - 1) / LANES;
                        const int osrc = og * LANES;
                        want &= want - 1u;
                        const bool mine = g == og;
                        const unsigned oa = __shfl_sync(PPG_FULL, a_off, osrc), ob = __shfl_sync(PPG_FULL, b_off, osrc);
                        const double o11 = shfl_d(i11, osrc), o12 = shfl_d(i12, osrc), o22 = shfl_d(i22, osrc);
                        const int omode = __shfl_sync(PPG_FULL, mode, osrc);
                        const unsigned ocoef = __shfl_sync(PPG_FULL, coef_sa, osrc);
                        const unsigned woff = (unsigned)lane * 8u;
                        double s[RW];
                        unsigned tb[RW];
#pragma unroll
                        for (int rr = 0; rr < RW; ++rr) {
                            const int r = rr * 32 + lane;
                            const double c = r < LD ? k2p_lds(ocoef + woff + rr * 256u) : 0.0;
                            tb[rr] = __ballot_sync(PPG_FULL, c != 0.0);
                            s[rr] = r < LD ? k2p_lds(v0_sa + woff + rr * 256u) : 0.0;
                        }
                        double ua = k2p_lds(v0_sa + oa), ub = has_b ? k2p_lds(v0_sa + ob) : 0.0;
#pragma unroll
                        for (int rr = 0; rr < RW; ++rr) {
                            unsigned bits = tb[rr];
                            while (bits) {
                                const unsigned jj = (unsigned)(rr * 32) + (unsigned)__ffs((int)bits) - 1u;
                                bits &= bits - 1u;
                                const double cj = k2p_lds(ocoef + jj * 8u);
                                const unsigned rb = gp_sa + jj * ROWB;
                                double gx[RW];
#pragma unroll
                                for (int r2 = 0; r2 < RW; ++r2) gx[r2] = r2 * 32 + lane < LD ? k2p_lds(rb + woff + r2 * 256u) : 0.0;
                                const double gxa = k2p_lds(rb + oa), gxb = k2p_lds(rb + ob);
#pragma unroll
                                for (int r2 = 0; r2 < RW; ++r2) s[r2] = fma(cj, gx[r2], s[r2]);
                                ua = fma(cj, gxa, ua);
                                ub = fma(cj, gxb, ub);
                            }
                        }
                        if (!has_b) ub = 0.0;
                        const double xa = -fma(o11, ua, o12 * ub), xb = -fma(o12, ua, o22 * ub);
                        const unsigned rpa = gp_sa + (oa >> 3) * ROWB + woff, rpb = gp_sa + (ob >> 3) * ROWB + woff;
                        double worst = 0.0, eqmax = 0.0, smax = 1.0;
                        bool fin = true;
#pragma unroll
                        for (int rr = 0; rr < RW; ++rr) {
                            const int r = rr * 32 + lane;
                            if (r < LD) s[rr] = fma(xa, k2p_lds(rpa + rr * 256u), fma(xb, k2p_lds(rpb + rr * 256u), s[rr]));
                            const bool pk = (r < P.mi && ((ctl.pf[(r >> 6) & 3] >> (r & 63)) & 1ull)) || (unsigned)r * 8u == oa ||
                                            (unsigned)r * 8u == ob;
                            if (r < R0) {
                                worst = fmax(worst, pk ? fabs(s[rr]) : s[rr]);
                                if (pk) eqmax = fmax(eqmax, fabs(s[rr]));
                                smax = fmax(smax, fabs(s[rr]));
                                fin = fin && fabs(s[rr]) < 1e300;
                            }
                        }
                        worst = warp_max_nonneg(worst);
                        fin = __all_sync(PPG_FULL, fin);
                        // hand-over only from a point whose residual vector is trustworthy (see oracle/twin.cpp k2p_certify):
                        // noise on the active rows = noise on every row; such candidates go to the simplex cold
                        // the active rows must hold as EQUALITIES, not merely within the LP tolerance (the simplex pivots them
                        // out exactly): a certificate, like a hand-over point, needs their residuals at rounding level
                        eqmax = warp_max_nonneg(eqmax);
                        smax = warp_max_nonneg(smax);
                        fin = fin && eqmax <= 1e-9 * smax;
                        const bool pass = omode == 1 && worst <= PPG_FEAS_TOL && fin;
                        bool again = false;
                        if (!pass && omode == 1) {
                            // converged by the running residuals but not by the exact ones: continue from the exact ones
                            const int rc = __shfl_sync(PPG_FULL, rechecks, osrc);
                            again = rc < 3;
                        }
                        const long long oidx = ctl.base + __shfl_sync(PPG_FULL, ci, osrc);
                        const uint8_t ost = (uint8_t)(__shfl_sync(PPG_FULL, cw, osrc) >> 24);
                        if (pass) {
                            if (lane == 0) { atomicAdd(&ctl.n_ok, 1ull); status[oidx] = ost | PPG_ST_FEAS; }
                            if (mine) have = false;
                        } else if (again) {
                            double* vs = scr_v + (size_t)warp * (RW * 32);
#pragma unroll
                            for (int rr = 0; rr < RW; ++rr) vs[rr * 32 + lane] = s[rr];
                            __syncwarp();
                            if (mine) {
#pragma unroll
                                for (int rr = 0; rr < RL; ++rr) v[rr] = ((park >> rr) & 1u) ? -1e300 : vs[rr * LANES + gl];
                                ++rechecks;
                                mode = 0;
                            }
                            __syncwarp();
                        } else {
                            if (P.warm_count != nullptr) {
                                // not certified: the last iterate becomes the simplex's origin (exact residuals)
                                unsigned long long slot = 0;
                                if (lane == 0) slot = atomicAdd(P.warm_count, 1ull);
                                slot = __shfl_sync(PPG_FULL, slot, 0);
                                if (slot < (unsigned long long)P.warm_cap) {
#pragma unroll
                                    for (int rr = 0; rr < RW; ++rr)
                                        if (fin && rr * 32 + lane < R0) P.warm_resid[slot * (unsigned long long)R0 + rr * 32 + lane] = s[rr];
                                    if (lane == 0) {
                                        P.warm_idx[slot] = fin ? oidx : -1;
                                        if (fin) status[oidx] = ost | PPG_ST_PRE;
                                    }
                                }
                            }
                            if (mine) have = false;
                        }
                        if (mine && !have) {
                            if (gl == 0) atomicAdd(&ctl.n_it, (unsigned long long)nst);
                            mode = 0;
                        }
                        __syncwarp();   // everybody is done reading the group's coefficients before its next set-up
                    }
                }
            }
            s0 = s1;
            __syncthreads();   // the segment's Gp and coefficient vectors are no longer read
        }
    }
    __syncthreads();
    if (tid == 0 && ctl.n_try) {
        atomicAdd(&counters[CNT_K2A_TRIED], ctl.n_try);
        atomicAdd(&counters[CNT_K2A_CERTIFIED], ctl.n_ok);
        atomicAdd(&counters[CNT_K2A_STEPS], ctl.n_it);
        atomicAdd(&counters[CNT_K2A_WORK], ctl.n_it * (unsigned long long)(R0 * (has_b ? 3 : 2)));
    }
}

template <int LANES, int RL, int THREADS>
static cudaError_t launch_k2p_t(const DevProgram& P, const uint64_t* masks, long long n, int k_act, uint8_t* status,
                                unsigned long long* queue, unsigned long long* counters, int max_iter, int sm_count,
                                cudaStream_t st, bool* handled) {
    constexpr int LD = RL * LANES;
    auto kern = k2p_relax_kernel<LANES, RL, THREADS>;
    const int p = k_act >= 2 ? k_act - 2 : 0;
    const size_t coef_d = (size_t)(THREADS / LANES) * LD;
    const size_t build_d = (size_t)2 * p * LD + (size_t)p * p;
    const size_t scratch = coef_d > build_d ? coef_d : build_d;
    const size_t smem = ((size_t)P.R0 * LD + LD + scratch) * sizeof(double) + (size_t)K2P_CHUNK * P.W * 8 + (size_t)K2P_CHUNK * 4 +
                        (size_t)(THREADS / 32) * ((LD + 31) / 32) * 32 * sizeof(double);
    if (smem > 220 * 1024) { *handled = false; return cudaSuccess; }
    cudaError_t e = allow_max_smem(kern);
    if (e != cudaSuccess) return e;
    int occ = 0;
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, THREADS, smem);
    if (e != cudaSuccess) return e;
    if (occ < 1) occ = 1;
    long long grid = (long long)sm_count * occ;
    // chunk: as large as staging allows while every CTA still sees several work items
    long long chunk = n / (grid * 8);
    if (chunk > K2P_CHUNK) chunk = K2P_CHUNK;
    if (chunk < 32) chunk = 32;
    const long long need = (n + chunk - 1) / chunk;
    if (grid > need) grid = need;
    if (grid < 1) grid = 1;
    static const int iters2 = getenv("PPGPU_K2A_ITERS2") ? atoi(getenv("PPGPU_K2A_ITERS2")) : 96;
    kern<<<(unsigned)grid, THREADS, smem, st>>>(P, masks, n, k_act, status, queue, counters, max_iter, iters2, (int)chunk,
                                                (int)scratch);
    *handled = true;
    return cudaGetLastError();
}

// returns cudaSuccess with *handled == false when the program is outside this kernel's envelope (the caller then uses
// the per-candidate kernels of k2a_relax.cu)
cudaError_t launch_k2a_prefix(const DevProgram& P, const uint64_t* masks, long long n, int k_act, uint8_t* status,
                              unsigned long long* queue, unsigned long long* counters, int max_iter, int sm_count,
                              cudaStream_t st, bool* handled) {
    *handled = false;
    static const int on = getenv("PPGPU_K2A_PREFIX") ? atoi(getenv("PPGPU_K2A_PREFIX")) : 1;
    if (!on || k_act < 1 || k_act - 2 > K2P_PMAX || P.R0 > 128 || P.W > 4) return cudaSuccess;
#define K2P_GO(L, R, T) return launch_k2p_t<L, R, T>(P, masks, n, k_act, status, queue, counters, max_iter, sm_count, st, handled)
    // 16 lanes x RL rows per candidate, 512 threads: measured best on the 100x30x6 program (8 lanes x 14 rows: fewer
    // instructions per candidate but 10 warps per SM hide less latency, 546 vs 488 ms; 640+ threads spill)
    static const int thr = getenv("PPGPU_K2P_THREADS") ? atoi(getenv("PPGPU_K2P_THREADS")) : 512;
    const int rh = (P.R0 + 15) / 16;
    if (rh == 7 && thr == 640) K2P_GO(16, 7, 640);
    if (rh == 7 && thr == 768) K2P_GO(16, 7, 768);
    switch (rh) {
        case 1: K2P_GO(16, 1, 512);
        case 2: K2P_GO(16, 2, 512);
        case 3: K2P_GO(16, 3, 512);
        case 4: K2P_GO(16, 4, 512);
        case 5: K2P_GO(16, 5, 512);
        case 6: K2P_GO(16, 6, 512);
        case 7: K2P_GO(16, 7, 512);
        default: K2P_GO(16, 8, 512);
    }
#undef K2P_GO
}

}  // namespace ppgpu
