// K2w - feasibility CERTIFICATES shared between the candidates of an enumeration level by walking over VERTICES.
//
// Question answered (per candidate active set A): is {z : g_r.z = h_r (r in A), g_r.z <= h_r (all r)} non-empty?
// (check_feasibility, /root/reference/src/ppopt/mplp_program.py:411-444 -> Solver.solve_lp, solver.py:211-246: one LP per
// candidate; mpqp_combinatorial.py:75-92 maps it over the level.)
//
// Observation: a feasible VERTEX v of F = {z : G z <= h} certifies EVERY candidate whose rows are all active at v - a
// nondegenerate vertex has nfree active rows, so it answers up to C(nfree, k') candidates of the level at once, while the
// relaxation of k2a_relax.cu / k2p_prefix.cu pays ~36 steps x R0 x 3 FMAs for each candidate separately (99.9 % of the
// candidates of the 100x30x6 program are feasible).  The level is in lexicographic order (mpqp_combinatorial.py:60-61),
// so the candidates that share their first k'-2 rows (the PREFIX) are contiguous; one warp ("walker") owns a chunk of the
// level and, prefix by prefix, moves a slack dictionary
//         s_B = beta - D s_N          (s = h - G z >= 0;  nonbasic slacks are 0: their rows are ACTIVE at the vertex)
// of the whole polyhedron F from vertex to vertex by primal simplex pivots:
//   drive(r): make row r nonbasic (active) while the rows in the FIXED set stay nonbasic - minimise s_r over the face of
//             the fixed rows: entering column = largest positive coefficient of row r, Harris ratio test, stop when r
//             leaves the basis.  Every vertex on the way is primal feasible.
//   segment (prefix P):  drive the rows of P one by one and fix them; then for every row a with open candidates: drive a,
//             fix it, and drive every b whose candidate P+{a,b} is still open.
//   after EVERY pivot the walker marks all open candidates P+{a,b} of the segment with a, b nonbasic: most candidates are
//             certified in passing (measured in a numpy model of this walk: 0.66 pivots per candidate at level 5).
// A certificate is therefore an exact statement: "the rows of A are nonbasic at a vertex whose basic slacks are >= -1e-8"
// (nonbasic slacks are zero by construction; beta carries the rounding of the pivots only: the dictionary is reloaded from
// the host-built vertex (host_math.hpp::build_walk_dictionary) at every work item and after K2W_RESET pivots).
// K2w never decides infeasibility and gives up freely (empty face, dependent row, iteration cap): whatever it leaves
// open goes to the relaxation (K2a) and then to the simplex (K2) exactly as before.
#include "common.cuh"
#include "launch.h"
#include "lp_core.cuh"

#include <cstdlib>

namespace ppgpu {

constexpr int K2W_MAXFIX = 30;      // longest prefix (k' - 2) the walker handles
constexpr int K2W_DRIVE_CAP = 400;  // pivots per drive before giving up
constexpr int K2W_RESET = 3000;     // pivots after which the dictionary is reloaded (bounds the accumulated rounding)
constexpr double K2W_PIV_MIN = 1e-7;   // smallest entering coefficient worth pivoting on
constexpr double K2W_NEG_OK = 1e-8;    // a vertex certifies only while every basic slack is >= -K2W_NEG_OK
// pivots K2wDeferDict keeps pending before it updates the whole dictionary (measured on the bench step, K2w 130.6 ms with
// every pivot applied to the whole dictionary: 117.3 at K = 2, 123.6 at 3, 138.2 at 4 - a longer pending chain on the
// entries a pivot reads costs more latency than the flushes it saves)
constexpr int K2W_DEFER = 2;

struct K2wCtx {
    double* D;        // nb x lds   [beta | coefficients], lds odd: rows over lanes are bank-conflict free
    double* prow;     // PROWS x lds scaled pivot row(s) of the storage policy
    int* bvar;        // nb         row id basic in dictionary row i
    int* nvar;        // nf         row id nonbasic in column j
    int* where;       // R0         >= 0: dictionary row, < 0: ~column
    uint64_t* orig;   // R0 x W4    segment: bit b >= a of row a = candidate P+{a,b} exists in the segment; bit a of row b (the
                      //             unused half) = ... and it passed the rank screen (only those may ever be certified)
    uint64_t* todo;   // R0 x W4    ... and is still open; symmetric (see k2w_mark_row)
    int* rowstart;    // R0         position in the segment of the first candidate with second-last row a
    uint64_t* nbm;    // W4         bitmask of the nonbasic rows
    int* fixrow;      // K2W_MAXFIX rows of the prefix currently fixed, in order
    uint64_t* witness; // n x PPG_WITNESS_SLOTS x Wm (global, may be null): nonbasic-row masks of vertices that hold a candidate
    int nb, nf, ld, lds, R0, W4, Wm;
};

__device__ __forceinline__ int k2w_top_bit(const uint64_t* m, int W, int* second) {
    int hi1 = -1, hi2 = -1;
    for (int w = W - 1; w >= 0 && hi2 < 0; --w) {
        uint64_t x = m[w];
        while (x && hi2 < 0) {
            const int t = w * 64 + 63 - __clzll((long long)x);
            x &= ~(1ull << (t & 63));
            if (hi1 < 0) hi1 = t; else hi2 = t;
        }
    }
    *second = hi2;
    return hi1;
}

// index of the j-th (0-based) set bit of a 4-word mask held in registers
__device__ __forceinline__ int k2w_nth(const uint64_t (&m)[4], int j) {
#pragma unroll
    for (int w = 0; w < 4; ++w) {
        const int cnt = __popcll(m[w]);
        if (j < cnt) {
            uint64_t x = m[w];
            for (int s = 0; s < j; ++s) x &= x - 1ull;
            return w * 64 + __ffsll((long long)x) - 1;
        }
        j -= cnt;
    }
    return -1;
}

// 1 / x to full double precision without the IEEE division sequence (x is a pivot / ratio denominator: normal, non-zero)
__device__ __forceinline__ double k2w_rcp(double x) {
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
    r = r * fma(-x, r, 2.0);
    return r * fma(-x, r, 2.0);
}

// labels of a Gauss-Jordan exchange (basic row l <-> nonbasic column j); lane 0
__device__ __forceinline__ void k2w_swap_labels(const K2wCtx& c, int l, int j) {
    const int rl = c.bvar[l], rn = c.nvar[j];
    c.bvar[l] = rn; c.nvar[j] = rl;
    c.where[rn] = l; c.where[rl] = ~j;
    c.nbm[rn >> 6] &= ~(1ull << (rn & 63));
    c.nbm[rl >> 6] |= 1ull << (rl & 63);
}

__device__ __forceinline__ void k2w_reload_labels(const DevProgram& P, const K2wCtx& c, int lane) {
    for (int w = lane; w < c.W4; w += 32) c.nbm[w] = 0ull;
    __syncwarp();
    for (int i = lane; i < c.nb; i += 32) { const int v = __ldg(P.wk_bvar + i); c.bvar[i] = v; c.where[v] = i; }
    for (int j = lane; j < c.nf; j += 32) {
        const int v = __ldg(P.wk_nvar + j);
        c.nvar[j] = v; c.where[v] = ~j;
        atomicOr(reinterpret_cast<unsigned long long*>(c.nbm + (v >> 6)), 1ull << (v & 63));
    }
    __syncwarp();
}

// ---- storage policy A: the dictionary in SHARED memory (any size that fits), lanes over rows
// LD_ > 0: the number of columns (wk_ld) is a compile-time constant (odd, so that it is its own row stride): the rank-1
// update unrolls into immediate-offset LDS / DFMA / STS with no bounds checks
template <int RPL_, int LD_ = 0>
struct K2wSmemDict {
    static constexpr int RPL = RPL_;
    static constexpr bool IN_SMEM = true;
    static constexpr int SMEM_ROW0 = 0;
    static constexpr int PROWS = 1;   // scaled pivot rows in shared memory (c.prow)
    __device__ __forceinline__ void reload(const DevProgram& P, const K2wCtx& c, int lane) {
        for (int e = lane; e < c.nb * c.ld; e += 32) {
            const int r = e / c.ld, k = e - r * c.ld;
            c.D[(size_t)r * c.lds + k] = __ldg(P.wk_D0 + e);
        }
        k2w_reload_labels(P, c, lane);
    }
    // right-hand side of basic row wi and its largest eligible coefficient (uniform results)
    __device__ __forceinline__ void target_scan(const K2wCtx& c, int wi, uint64_t fm, int lane, double& bi, double& wbest, int& j) {
        const int lds = LD_ > 0 ? LD_ : c.lds;
        const double* Di = c.D + (size_t)wi * lds;
        bi = Di[0];
        const bool degen = bi <= 1e-11;
        double best = 0.0; int bj = 0x7fffffff;
        for (int jj = lane; jj < c.nf; jj += 32) {
            if ((fm >> jj) & 1ull) continue;
            double x = Di[1 + jj];
            if (degen) x = fabs(x);
            if (x > best) { best = x; bj = jj; }
        }
        wbest = warp_max_nonneg(best);
        j = __reduce_min_sync(PPG_FULL, best == wbest ? bj : 0x7fffffff);
    }
    __device__ __forceinline__ void column(const K2wCtx& c, int j, int lane, double (&col)[RPL], double (&beta)[RPL]) {
#pragma unroll
        for (int rr = 0; rr < RPL; ++rr) {
            const int r = lane + 32 * rr;
            const int lds = LD_ > 0 ? LD_ : c.lds;
            col[rr] = r < c.nb ? c.D[(size_t)r * lds + 1 + j] : 0.0;
            beta[rr] = r < c.nb ? c.D[(size_t)r * lds] : 0.0;
        }
    }
    // basic row l leaves, nonbasic column j enters.  Returns false (uniformly) when some basic slack ends below -K2W_NEG_OK.
    __device__ __forceinline__ bool pivot(const K2wCtx& c, int l, int j, int lane) {
        const int cj = 1 + j, lds = LD_ > 0 ? LD_ : c.lds, ld = LD_ > 0 ? LD_ : c.ld, nb = c.nb;
        double* Dl = c.D + (size_t)l * lds;
        const double inv = k2w_rcp(Dl[cj]);
        __syncwarp();
        for (int k = lane; k < ld; k += 32) c.prow[k] = (k == cj) ? 0.0 : Dl[k] * inv;
        __syncwarp();
        double colr[RPL];
        double* Dr[RPL];
#pragma unroll
        for (int rr = 0; rr < RPL; ++rr) {
            const int r = lane + 32 * rr;
            Dr[rr] = c.D + (size_t)(r < nb ? r : 0) * lds;
            colr[rr] = (r < nb && r != l) ? Dr[rr][cj] : 0.0;
        }
        const double* __restrict__ q = c.prow;
        // rank-1 update in groups of G columns: every load of a group is issued before its first FMA (the compiler cannot
        // hoist a shared-memory load above a store to another row on its own: one exposed LDS latency per element otherwise)
        constexpr int G = 8;
        bool okb = true;
        if constexpr (LD_ > 0) {
            static_for<(LD_ + G - 1) / G>([&](auto KK) {
                constexpr int k0 = decltype(KK)::value * G;
                constexpr int GN = (LD_ - k0) < G ? (LD_ - k0) : G;
                double qk[GN], x[RPL][GN];
#pragma unroll
                for (int g = 0; g < GN; ++g) qk[g] = q[k0 + g];
#pragma unroll
                for (int rr = 0; rr < RPL; ++rr)
#pragma unroll
                    for (int g = 0; g < GN; ++g) x[rr][g] = Dr[rr][k0 + g];
#pragma unroll
                for (int rr = 0; rr < RPL; ++rr)
#pragma unroll
                    for (int g = 0; g < GN; ++g) x[rr][g] = fma(-colr[rr], qk[g], x[rr][g]);
                if constexpr (k0 == 0) {
                    // column 0 is the right-hand side: the certification band is checked on the value just computed
#pragma unroll
                    for (int rr = 0; rr < RPL; ++rr) {
                        const int r = lane + 32 * rr;
                        okb = okb && (r >= nb || r == l || x[rr][0] >= -K2W_NEG_OK);
                    }
                }
#pragma unroll
                for (int rr = 0; rr < RPL; ++rr)
                    if (colr[rr] != 0.0) {
#pragma unroll
                        for (int g = 0; g < GN; ++g) Dr[rr][k0 + g] = x[rr][g];
                    }
            });
        } else {
            for (int k0 = 0; k0 < ld; k0 += G) {
                double qk[G], x[RPL][G];
#pragma unroll
                for (int g = 0; g < G; ++g) qk[g] = (k0 + g < ld) ? q[k0 + g] : 0.0;
#pragma unroll
                for (int rr = 0; rr < RPL; ++rr)
#pragma unroll
                    for (int g = 0; g < G; ++g) x[rr][g] = (k0 + g < ld) ? Dr[rr][k0 + g] : 0.0;
#pragma unroll
                for (int rr = 0; rr < RPL; ++rr)
#pragma unroll
                    for (int g = 0; g < G; ++g) x[rr][g] = fma(-colr[rr], qk[g], x[rr][g]);
#pragma unroll
                for (int rr = 0; rr < RPL; ++rr)
                    if (colr[rr] != 0.0) {
#pragma unroll
                        for (int g = 0; g < G; ++g)
                            if (k0 + g < ld) Dr[rr][k0 + g] = x[rr][g];
                    }
            }
        }
        bool ok = okb;
#pragma unroll
        for (int rr = 0; rr < RPL; ++rr) {
            const int r = lane + 32 * rr;
            if (r < nb && r != l) {
                if (colr[rr] != 0.0) Dr[rr][cj] = -colr[rr] * inv;
                if constexpr (LD_ == 0) ok = ok && Dr[rr][0] >= -K2W_NEG_OK;
            }
        }
        __syncwarp();
        for (int k = lane; k < ld; k += 32) Dl[k] = (k == cj) ? inv : q[k];
        if (lane == 0) k2w_swap_labels(c, l, j);
        ok = __all_sync(PPG_FULL, ok);
        __syncwarp();
        return ok;
    }
};

// ---- storage policy D: the dictionary in SHARED memory with DEFERRED updates - policy A's arithmetic, bit for bit, but
// the rank-1 updates reach the bulk of D only once every K pivots.  Per pending step m the walker keeps the scaled pivot
// row p_m (c.prow + m * LD: policy A's prow, 0 in the entering column cj_m) and, in registers, u_m[r] = policy A's colr
// (the entering-column entry of row r, 0 for the pivot row and rows >= nb).  The current value of entry (i, k) is
//         D[i][k], then x = fma(-u_m[i], p_m[k], x) for every pending m in order
// - the FMAs policy A performs, in the same order.  The two overwrites of a Gauss-Jordan step are stored at once and
// cancel the pending steps on what they overwrite: the new pivot row goes straight into D and its owner zeroes u_m'[l],
// the exchanged column -u_m[r] / pivot goes into D for every other row and p_m'[cj] = 0 (m' < m).  Only signs of zeros
// can differ from policy A, which no comparison observes.  The right-hand side (column 0) lives in registers and is
// updated at every pivot like policy A's column 0, so the certification band is still checked after every pivot;
// column 0 of D is only read by reload.  Per pivot (76 x 37) this reads / writes ~3.2 k dictionary entries at K = 2
// (~1.8 k at K = 4) instead of ~5.6 k: the target row, the entering column and the pivot row through the pending chain,
// plus 1 / K of a flush.
template <int RPL_, int LD, int K>
struct K2wDeferDict {
    static constexpr int RPL = RPL_;
    static constexpr bool IN_SMEM = true;
    static constexpr int SMEM_ROW0 = 0;
    static constexpr int PROWS = K;
    double u[K][RPL];   // u_m of my rows (lane + 32 rr)
    double beta[RPL];   // right-hand side of my rows, always current
    int np;             // pending steps (uniform); np == pivots since reload mod K
    // current values the next pivot may reuse: row trow_i at columns 1 + lane + 32 h (target_scan), the entering column
    // 1 + ccol_j of my rows (column)
    static constexpr int TH = (LD - 1 + 31) / 32;
    double trow[TH], ccol[RPL];
    int trow_i, ccol_j;
    // value of basic row `slot * 32 + owner`, uniform over the warp
    template <int N>
    __device__ __forceinline__ double from_row(const double (&v)[N], int slot, int owner) const {
        double x = 0.0;
#pragma unroll
        for (int rr = 0; rr < N; ++rr) if (rr == slot) x = v[rr];
        return shfl_d(x, owner);
    }
    // u_m of basic row l (uniform), m < np
    __device__ __forceinline__ void row_u(int l, double (&ul)[K]) const {
#pragma unroll
        for (int m = 0; m < K; ++m) ul[m] = m < np ? from_row(u[m], l >> 5, l & 31) : 0.0;
    }
    // current value of an entry from its stored value: the pending chain with row factors um, column k of the p_m
    __device__ __forceinline__ double chain(const K2wCtx& c, double x, const double (&um)[K], int k) const {
#pragma unroll
        for (int m = 0; m < K; ++m)
            if (m < np) x = fma(-um[m], c.prow[m * LD + k], x);
        return x;
    }
    __device__ __forceinline__ void reload(const DevProgram& P, const K2wCtx& c, int lane) {
        for (int e = lane; e < c.nb * LD; e += 32) c.D[e] = __ldg(P.wk_D0 + e);
#pragma unroll
        for (int rr = 0; rr < RPL; ++rr) {
            const int r = lane + 32 * rr;
            beta[rr] = r < c.nb ? __ldg(P.wk_D0 + (size_t)r * LD) : 0.0;
        }
        np = 0;   // whatever was pending is discarded with the old dictionary
        trow_i = -1; ccol_j = -1;
        k2w_reload_labels(P, c, lane);
    }
    __device__ __forceinline__ void target_scan(const K2wCtx& c, int wi, uint64_t fm, int lane, double& bi, double& wbest, int& j) {
        double uw[K];
        row_u(wi, uw);
        bi = from_row(beta, wi >> 5, wi & 31);
        const double* Di = c.D + (size_t)wi * LD;
        const bool degen = bi <= 1e-11;
        double best = 0.0; int bj = 0x7fffffff;
#pragma unroll
        for (int h = 0; h < TH; ++h) {
            const int jj = lane + 32 * h;
            if (1 + jj >= LD) continue;
            trow[h] = chain(c, Di[1 + jj], uw, 1 + jj);
            if (jj >= c.nf || ((fm >> jj) & 1ull)) continue;
            const double x = degen ? fabs(trow[h]) : trow[h];
            if (x > best) { best = x; bj = jj; }
        }
        trow_i = wi;
        wbest = warp_max_nonneg(best);
        j = __reduce_min_sync(PPG_FULL, best == wbest ? bj : 0x7fffffff);
    }
    // entering column of my rows (lanes over rows, broadcast loads of p_m[cj])
    __device__ __forceinline__ void cur_column(const K2wCtx& c, int cj, int lane, double (&col)[RPL]) const {
#pragma unroll
        for (int rr = 0; rr < RPL; ++rr) {
            const int r = lane + 32 * rr;
            double um[K];
#pragma unroll
            for (int m = 0; m < K; ++m) um[m] = u[m][rr];
            col[rr] = r < c.nb ? chain(c, c.D[(size_t)r * LD + cj], um, cj) : 0.0;
        }
    }
    __device__ __forceinline__ void column(const K2wCtx& c, int j, int lane, double (&col)[RPL], double (&beta_out)[RPL]) {
        cur_column(c, 1 + j, lane, col);
#pragma unroll
        for (int rr = 0; rr < RPL; ++rr) { ccol[rr] = col[rr]; beta_out[rr] = beta[rr]; }
        ccol_j = j;
    }
    __device__ __forceinline__ bool pivot(const K2wCtx& c, int l, int j, int lane) {
        const int cj = 1 + j, nb = c.nb, slot = l >> 5, owner = l & 31;
        double col[RPL];
        if (ccol_j == j) {
#pragma unroll
            for (int rr = 0; rr < RPL; ++rr) col[rr] = ccol[rr];
        } else {
            cur_column(c, cj, lane, col);
        }
        const double inv = k2w_rcp(from_row(col, slot, owner));
        double ul[K];
        row_u(l, ul);
        const double q0 = from_row(beta, slot, owner) * inv;
        __syncwarp();
        // the pivot row: p_np = current row l x inv (0 in the entering column), and the new row l stored in D
        double* Dl = c.D + (size_t)l * LD;
        double* pn = c.prow + np * LD;
        if (lane == 0) pn[0] = q0;
#pragma unroll
        for (int h = 0; h < TH; ++h) {
            const int k = 1 + lane + 32 * h;
            if (k >= LD) continue;
            const double x = trow_i == l ? trow[h] : chain(c, Dl[k], ul, k);
            const double q = (k == cj) ? 0.0 : x * inv;
            pn[k] = q;
            Dl[k] = (k == cj) ? inv : q;
        }
        trow_i = -1; ccol_j = -1;
        bool ok = true;
#pragma unroll
        for (int rr = 0; rr < RPL; ++rr) {
            const int r = lane + 32 * rr;
            if (r == l) {
                // the new row l carries none of the earlier pending steps
#pragma unroll
                for (int m = 0; m < K; ++m) if (m < np) u[m][rr] = 0.0;
            }
            const double ur = (r < nb && r != l) ? col[rr] : 0.0;
#pragma unroll
            for (int m = 0; m < K; ++m) if (m == np) u[m][rr] = ur;
            // right-hand side: policy A's column 0, checked on the value just computed
            const double x = fma(-ur, q0, beta[rr]);
            beta[rr] = r == l ? q0 : x;
            ok = ok && (r >= nb || r == l || x >= -K2W_NEG_OK);
            // the exchanged column, stored for every other row (zeros included: the earlier steps are cancelled on it)
            if (r < nb && r != l) c.D[(size_t)r * LD + cj] = -ur * inv;
        }
        __syncwarp();
        if (lane < np) c.prow[lane * LD + cj] = 0.0;
        if (lane == 0) k2w_swap_labels(c, l, j);
        if (++np == K) {
            __syncwarp();
            flush(c, lane);
        }
        ok = __all_sync(PPG_FULL, ok);
        __syncwarp();
        return ok;
    }
    // the K pending steps applied to columns 1.. of every row: one load, K FMAs and one store per entry, in groups of G
    // columns whose loads are all issued before their first FMA (as policy A's update).  A row whose pending u are all zero
    // is not stored (policy A skips the store of a row whose column entry is zero).
    __device__ __forceinline__ void flush(const K2wCtx& c, int lane) {
        constexpr int G = 6;
        double* Dr[RPL];
        bool st[RPL];
#pragma unroll
        for (int rr = 0; rr < RPL; ++rr) {
            const int r = lane + 32 * rr;
            Dr[rr] = c.D + (size_t)(r < c.nb ? r : 0) * LD;
            st[rr] = false;
#pragma unroll
            for (int m = 0; m < K; ++m) st[rr] = st[rr] || u[m][rr] != 0.0;
        }
        const double* __restrict__ p = c.prow;
        static_for<(LD - 1 + G - 1) / G>([&](auto KK) {
            constexpr int k0 = 1 + decltype(KK)::value * G;
            constexpr int GN = (LD - k0) < G ? (LD - k0) : G;
            double x[RPL][GN];
#pragma unroll
            for (int rr = 0; rr < RPL; ++rr)
#pragma unroll
                for (int g = 0; g < GN; ++g) x[rr][g] = Dr[rr][k0 + g];
#pragma unroll
            for (int m = 0; m < K; ++m) {
                double pk[GN];
#pragma unroll
                for (int g = 0; g < GN; ++g) pk[g] = p[m * LD + k0 + g];
#pragma unroll
                for (int rr = 0; rr < RPL; ++rr)
#pragma unroll
                    for (int g = 0; g < GN; ++g) x[rr][g] = fma(-u[m][rr], pk[g], x[rr][g]);
            }
#pragma unroll
            for (int rr = 0; rr < RPL; ++rr)
                if (st[rr]) {
#pragma unroll
                    for (int g = 0; g < GN; ++g) Dr[rr][k0 + g] = x[rr][g];
                }
        });
        np = 0;
    }
};

// ---- storage policy C: HYBRID - the first 32 basic rows (row slot 0: one row per lane) in REGISTERS, the other slots in
// shared memory.  The walk is bound by shared-memory bandwidth (a pivot reads and writes every dictionary entry: ncu 69 %
// of the wavefront peak with everything in shared memory); one slot in registers removes 4 of the 11 wavefronts per column
// of the rank-1 update while the register count stays where it is (LD doubles more per thread: no spills, unlike the
// all-register policy B).  LD = wk_ld exactly (compile-time, odd).  Register arrays are only indexed by constants
// (static_for / reg_pick / reg_set).
template <int RPL_, int LD>
struct K2wHybridDict {
    static constexpr int RPL = RPL_;
    static constexpr bool IN_SMEM = true;
    static constexpr int SMEM_ROW0 = 32;   // shared memory holds rows 32.. (row r at (r - 32) * LD)
    static constexpr int PROWS = 1;
    double T0[LD];                          // row `lane` of the dictionary
    __device__ __forceinline__ void reload(const DevProgram& P, const K2wCtx& c, int lane) {
#pragma unroll
        for (int k = 0; k < LD; ++k) T0[k] = lane < c.nb ? __ldg(P.wk_D0 + (size_t)lane * LD + k) : 0.0;
        for (int e = lane + 32 * LD; e < c.nb * LD; e += 32) c.D[e - 32 * LD] = __ldg(P.wk_D0 + e);
        k2w_reload_labels(P, c, lane);
    }
    __device__ __forceinline__ void target_scan(const K2wCtx& c, int wi, uint64_t fm, int lane, double& bi, double& wbest, int& j) {
        if (wi < 32) {
            // the owner lane scans its own registers, the result is broadcast
            const double b0 = T0[0];
            const bool degen = b0 <= 1e-11;
            double best = 0.0; int bj = 0x7fffffff;
#pragma unroll
            for (int k = 1; k < LD; ++k) {
                double x = T0[k];
                if (degen) x = fabs(x);
                if (!((fm >> (k - 1)) & 1ull) && x > best) { best = x; bj = k - 1; }
            }
            bi = shfl_d(b0, wi);
            wbest = shfl_d(best, wi);
            j = __shfl_sync(PPG_FULL, bj, wi);
        } else {
            const double* Di = c.D + (size_t)(wi - 32) * LD;
            bi = Di[0];
            const bool degen = bi <= 1e-11;
            double best = 0.0; int bj = 0x7fffffff;
            for (int jj = lane; jj < c.nf; jj += 32) {
                if ((fm >> jj) & 1ull) continue;
                double x = Di[1 + jj];
                if (degen) x = fabs(x);
                if (x > best) { best = x; bj = jj; }
            }
            wbest = warp_max_nonneg(best);
            j = __reduce_min_sync(PPG_FULL, best == wbest ? bj : 0x7fffffff);
        }
    }
    __device__ __forceinline__ void column(const K2wCtx& c, int j, int lane, double (&col)[RPL], double (&beta)[RPL]) {
        col[0] = lane < c.nb ? reg_pick<LD>(T0, 1 + j) : 0.0;
        beta[0] = T0[0];
#pragma unroll
        for (int rr = 1; rr < RPL; ++rr) {
            const int r = lane + 32 * rr;
            col[rr] = r < c.nb ? c.D[(size_t)(r - 32) * LD + 1 + j] : 0.0;
            beta[rr] = r < c.nb ? c.D[(size_t)(r - 32) * LD] : 0.0;
        }
    }
    __device__ __forceinline__ bool pivot(const K2wCtx& c, int l, int j, int lane) {
        const int cj = 1 + j, nb = c.nb;
        const bool l_in_regs = l < 32;
        double* Dl = c.D + (size_t)(l_in_regs ? 0 : l - 32) * LD;
        const double c0 = reg_pick<LD>(T0, cj);       // my register row's entry in the entering column
        const double piv = l_in_regs ? shfl_d(c0, l) : Dl[cj];
        const double inv = k2w_rcp(piv);
        __syncwarp();
        if (l_in_regs) {
            if (lane == l) {
#pragma unroll
                for (int k = 0; k < LD; ++k) c.prow[k] = T0[k] * inv;
                c.prow[cj] = 0.0;
            }
        } else {
            for (int k = lane; k < LD; k += 32) c.prow[k] = (k == cj) ? 0.0 : Dl[k] * inv;
        }
        __syncwarp();
        double colr[RPL];
        double* Dr[RPL];
        colr[0] = (lane < nb && lane != l) ? c0 : 0.0;
        Dr[0] = nullptr;
#pragma unroll
        for (int rr = 1; rr < RPL; ++rr) {
            const int r = lane + 32 * rr;
            Dr[rr] = c.D + (size_t)(r < nb ? r - 32 : 0) * LD;
            colr[rr] = (r < nb && r != l) ? Dr[rr][cj] : 0.0;
        }
        const double* __restrict__ q = c.prow;
        const bool own = l_in_regs && lane == l;
        constexpr int G = 8;
        bool okb = true;
        static_for<(LD + G - 1) / G>([&](auto KK) {
            constexpr int k0 = decltype(KK)::value * G;
            constexpr int GN = (LD - k0) < G ? (LD - k0) : G;
            double qk[GN], x[RPL][GN];
#pragma unroll
            for (int g = 0; g < GN; ++g) qk[g] = q[k0 + g];
#pragma unroll
            for (int rr = 1; rr < RPL; ++rr)
#pragma unroll
                for (int g = 0; g < GN; ++g) x[rr][g] = Dr[rr][k0 + g];
            // slot 0: registers; the pivot row's owner takes the scaled row itself
#pragma unroll
            for (int g = 0; g < GN; ++g) {
                const double v = fma(-colr[0], qk[g], T0[k0 + g]);
                T0[k0 + g] = own ? qk[g] : v;
            }
#pragma unroll
            for (int rr = 1; rr < RPL; ++rr)
#pragma unroll
                for (int g = 0; g < GN; ++g) x[rr][g] = fma(-colr[rr], qk[g], x[rr][g]);
            if constexpr (k0 == 0) {
                okb = okb && (lane >= nb || lane == l || T0[0] >= -K2W_NEG_OK);
#pragma unroll
                for (int rr = 1; rr < RPL; ++rr) {
                    const int r = lane + 32 * rr;
                    okb = okb && (r >= nb || r == l || x[rr][0] >= -K2W_NEG_OK);
                }
            }
#pragma unroll
            for (int rr = 1; rr < RPL; ++rr)
                if (colr[rr] != 0.0) {
#pragma unroll
                    for (int g = 0; g < GN; ++g) Dr[rr][k0 + g] = x[rr][g];
                }
        });
        // the exchanged column: -col / pivot for the other rows, 1 / pivot for the pivot row
        reg_set<LD>(T0, cj, own ? inv : -colr[0] * inv);
#pragma unroll
        for (int rr = 1; rr < RPL; ++rr) {
            const int r = lane + 32 * rr;
            if (r < nb && r != l && colr[rr] != 0.0) Dr[rr][cj] = -colr[rr] * inv;
        }
        __syncwarp();
        if (!l_in_regs)
            for (int k = lane; k < LD; k += 32) Dl[k] = (k == cj) ? inv : q[k];
        if (lane == 0) k2w_swap_labels(c, l, j);
        const bool ok = __all_sync(PPG_FULL, okb);
        __syncwarp();
        return ok;
    }
};

// ---- storage policy B: the dictionary in REGISTERS - lane (r & 31) holds basic row r in slot r >> 5, DC = columns incl.
// the right-hand side (exactly wk_ld).  Only the scaled pivot row crosses shared memory (DC doubles per pivot); the rank-1
// update is RPL x DC back-to-back DFMAs on registers.  Register arrays are only ever indexed by compile-time constants
// (static_for / reg_pick / reg_set of lp_core.cuh), else the dictionary would fall into local memory.
template <int RPL_, int DC>
struct K2wRegDict {
    static constexpr int RPL = RPL_;
    static constexpr bool IN_SMEM = false;
    static constexpr int SMEM_ROW0 = 0;
    static constexpr int PROWS = 1;
    double T[RPL][DC];
    __device__ __forceinline__ void reload(const DevProgram& P, const K2wCtx& c, int lane) {
        static_for<RPL>([&](auto RR) {
            constexpr int rr = decltype(RR)::value;
            const int r = lane + 32 * rr;
#pragma unroll
            for (int k = 0; k < DC; ++k) T[rr][k] = r < c.nb ? __ldg(P.wk_D0 + (size_t)r * DC + k) : 0.0;
        });
        k2w_reload_labels(P, c, lane);
    }
    __device__ __forceinline__ void target_scan(const K2wCtx& c, int wi, uint64_t fm, int lane, double& bi, double& wbest, int& j) {
        // the owner lane scans its own row (no shared-memory round trip), the result is broadcast
        const int slot = wi >> 5, owner = wi & 31;
        double b0 = 0.0, best = 0.0; int bj = 0x7fffffff;
        static_for<RPL>([&](auto RR) {
            constexpr int rr = decltype(RR)::value;
            if (rr == slot) {
                b0 = T[rr][0];
                const bool degen = b0 <= 1e-11;
#pragma unroll
                for (int k = 1; k < DC; ++k) {
                    double x = T[rr][k];
                    if (degen) x = fabs(x);
                    if (!((fm >> (k - 1)) & 1ull) && x > best) { best = x; bj = k - 1; }
                }
            }
        });
        bi = shfl_d(b0, owner);
        wbest = shfl_d(best, owner);
        j = __shfl_sync(PPG_FULL, bj, owner);
    }
    __device__ __forceinline__ void column(const K2wCtx& c, int j, int lane, double (&col)[RPL], double (&beta)[RPL]) {
        static_for<RPL>([&](auto RR) {
            constexpr int rr = decltype(RR)::value;
            col[rr] = (lane + 32 * rr < c.nb) ? reg_pick<DC>(T[rr], 1 + j) : 0.0;
            beta[rr] = T[rr][0];
        });
    }
    __device__ __forceinline__ bool pivot(const K2wCtx& c, int l, int j, int lane) {
        const int cj = 1 + j, slot = l >> 5, owner = l & 31, nb = c.nb;
        double colr[RPL];
        static_for<RPL>([&](auto RR) {
            constexpr int rr = decltype(RR)::value;
            colr[rr] = reg_pick<DC>(T[rr], cj);
        });
        double piv = 0.0;
        static_for<RPL>([&](auto RR) {
            constexpr int rr = decltype(RR)::value;
            if (rr == slot) piv = colr[rr];
        });
        const double inv = k2w_rcp(shfl_d(piv, owner));
        __syncwarp();
        static_for<RPL>([&](auto RR) {
            constexpr int rr = decltype(RR)::value;
            if (rr == slot && lane == owner) {
#pragma unroll
                for (int k = 0; k < DC; ++k) c.prow[k] = T[rr][k] * inv;
                c.prow[cj] = 0.0;
            }
        });
        __syncwarp();
        const double* __restrict__ q = c.prow;
        static_for<RPL>([&](auto RR) {
            constexpr int rr = decltype(RR)::value;
            const int r = lane + 32 * rr;
            if (r >= nb || r == l) colr[rr] = 0.0;
        });
        bool ok = true;
#pragma unroll
        for (int k = 0; k < DC; ++k) {
            const double qk = q[k];
            static_for<RPL>([&](auto RR) {
                constexpr int rr = decltype(RR)::value;
                T[rr][k] = fma(-colr[rr], qk, T[rr][k]);
            });
        }
        static_for<RPL>([&](auto RR) {
            constexpr int rr = decltype(RR)::value;
            const int r = lane + 32 * rr;
            if (r == l) {
                // the pivot row itself: the scaled row, 1 / pivot in the exchanged column
#pragma unroll
                for (int k = 0; k < DC; ++k) T[rr][k] = q[k];
                reg_set<DC>(T[rr], cj, inv);
            } else {
                reg_set<DC>(T[rr], cj, -colr[rr] * inv);   // (rows beyond nb and zero entries: stays 0)
                ok = ok && (r >= nb || T[rr][0] >= -K2W_NEG_OK);
            }
        });
        if (lane == 0) k2w_swap_labels(c, l, j);
        ok = __all_sync(PPG_FULL, ok);
        __syncwarp();
        return ok;
    }
};

// bits of word w with index >= a
__device__ __forceinline__ uint64_t k2w_ge_mask(int a, int w) {
    const int aw = a >> 6;
    return w < aw ? 0ull : (w == aw ? (~0ull << (a & 63)) : ~0ull);
}

// certify candidate (a, b) of the segment (the caller has cleared its todo bit)
__device__ __forceinline__ void k2w_certify(const K2wCtx& c, uint8_t* __restrict__ status, long long seg_base, int a, int b) {
    int rank = 0;
    const int w = b >> 6;
    for (int w2 = 0; w2 < w; ++w2) rank += __popcll(c.orig[(size_t)a * c.W4 + w2] & k2w_ge_mask(a, w2));
    rank += __popcll(c.orig[(size_t)a * c.W4 + w] & k2w_ge_mask(a, w) & ((1ull << (b & 63)) - 1ull));
    const long long idx = seg_base + c.rowstart[a] + rank;
    // fire-and-forget OR on the aligned word that holds the byte (a load + store would stall the walker for an L2 round trip)
    const uintptr_t addr = reinterpret_cast<uintptr_t>(status + idx);
    atomicOr(reinterpret_cast<unsigned*>(addr & ~(uintptr_t)3), (unsigned)PPG_ST_FEAS << (8u * (unsigned)(addr & 3)));
    // the WITNESS: the rows active at the certifying vertex.  Every superset of the candidate inside this mask is certified
    // by the same vertex - the next level inherits it (k6_children.cu::inherit_kernel) instead of walking again
    if (c.witness)
        for (int w = 0; w < c.Wm; ++w) c.witness[idx * (PPG_WITNESS_SLOTS * c.Wm) + w] = c.nbm[w];
}

// second witness slot of candidate (a, b), a < b, which is closed already: the vertex the walk is at holds it as well.
// Two different vertices per parent cover more children than one (CPU model, level 4 -> 5 of the 100x30x6 program: 76 % of
// the children inherit from first witnesses alone, 88 % with a later vertex next to them)
__device__ __forceinline__ void k2w_second_witness(const K2wCtx& c, uint8_t* __restrict__ status, long long seg_base, int a, int b, int turn) {
    int rank = 0;
    const int w = b >> 6;
    for (int w2 = 0; w2 < w; ++w2) rank += __popcll(c.orig[(size_t)a * c.W4 + w2] & k2w_ge_mask(a, w2));
    rank += __popcll(c.orig[(size_t)a * c.W4 + w] & k2w_ge_mask(a, w) & ((1ull << (b & 63)) - 1ull));
    const long long idx = seg_base + c.rowstart[a] + rank;
    const int slot = 1 + (turn % (PPG_WITNESS_SLOTS - 1));
    for (int x = 0; x < c.Wm; ++x) c.witness[idx * (PPG_WITNESS_SLOTS * c.Wm) + slot * c.Wm + x] = c.nbm[x];
    // (a candidate the walk gave up on earlier is closed too; its feasible bit is left to the relaxation / the simplex, and
    // its witness is only ever used if they set it: the next level looks at the witnesses of FEASIBLE parents)
    (void)status;
}

// after a pivot that made row r nonbasic (and after k2w_mark_row): every CLOSED candidate {r, y} of the segment with y
// nonbasic is revisited; lanes over y.  (Measured on the bench program: revisiting only one block of 32 rows y per pivot
// makes level 4 cheaper but leaves older second witnesses - 81.5 % of level 5 inherit instead of 85.5 %, the step is 8 ms
// slower.)
__device__ __forceinline__ void k2w_revisit_row(const K2wCtx& c, uint8_t* __restrict__ status, long long seg_base, int r, int lane, int turn) {
    for (int y = lane; y < c.R0; y += 32) {
        if (y == r || !((c.nbm[y >> 6] >> (y & 63)) & 1ull)) continue;
        const int a = y < r ? y : r, b = y < r ? r : y;
        const uint64_t bit = 1ull << (b & 63);
        if (!(c.orig[(size_t)a * c.W4 + (b >> 6)] & bit) || (c.todo[(size_t)a * c.W4 + (b >> 6)] & bit)) continue;
        if (!((c.orig[(size_t)b * c.W4 + (a >> 6)] >> (a & 63)) & 1ull)) continue;   // failed the rank screen
        k2w_second_witness(c, status, seg_base, a, b, turn);
    }
}

// the same for every closed candidate at the first vertex of a segment (the prefix has just been fixed); lanes over a
__device__ __forceinline__ void k2w_revisit_all(const K2wCtx& c, uint8_t* __restrict__ status, long long seg_base, int lane) {
    for (int a = lane; a < c.R0; a += 32) {
        if (!((c.nbm[a >> 6] >> (a & 63)) & 1ull)) continue;
        for (int w = 0; w < c.W4; ++w) {
            uint64_t bits = c.nbm[w] & c.orig[(size_t)a * c.W4 + w] & ~c.todo[(size_t)a * c.W4 + w] & k2w_ge_mask(a + 1, w);
            while (bits) {
                const int bb = w * 64 + __ffsll((long long)bits) - 1;
                bits &= bits - 1ull;
                if (!((c.orig[(size_t)bb * c.W4 + (a >> 6)] >> (a & 63)) & 1ull)) continue;   // failed the rank screen
                k2w_second_witness(c, status, seg_base, a, bb, 0);
            }
        }
    }
}

// Open candidates live in a SYMMETRIC bit matrix: bit y of row x is set while the candidate with last rows {x, y} is open
// (single-row candidates: the diagonal).  The half with y >= x is canonical, the other half mirrors it so that "which open
// candidates does row r belong to" is ONE row read (the mirror may lag behind: it is confirmed against the canonical bit).

// marks every open candidate of the segment whose last two rows are nonbasic (full scan: after the prefix is fixed)
__device__ __forceinline__ int k2w_mark_all(const K2wCtx& c, uint8_t* __restrict__ status, long long seg_base, int lane) {
    int got = 0;
    for (int a = lane; a < c.R0; a += 32) {
        if (!((c.nbm[a >> 6] >> (a & 63)) & 1ull)) continue;
        for (int w = 0; w < c.W4; ++w) {
            uint64_t bits = c.nbm[w] & c.todo[(size_t)a * c.W4 + w] & k2w_ge_mask(a, w);
            if (!bits) continue;
            atomicAnd(reinterpret_cast<unsigned long long*>(c.todo + (size_t)a * c.W4 + w), ~bits);
            while (bits) {
                const int bb = w * 64 + __ffsll((long long)bits) - 1;
                bits &= bits - 1ull;
                if (bb != a) atomicAnd(reinterpret_cast<unsigned long long*>(c.todo + (size_t)bb * c.W4 + (a >> 6)), ~(1ull << (a & 63)));
                k2w_certify(c, status, seg_base, a, bb);
                ++got;
            }
        }
    }
    return got;
}

// after a pivot only the candidates with the row r that has just become nonbasic can be new: one read of row r
__device__ __forceinline__ int k2w_mark_row(const K2wCtx& c, uint8_t* __restrict__ status, long long seg_base, int r, int lane) {
    int got = 0;
    for (int w = 0; w < c.W4; ++w) {
        uint64_t bits = c.todo[(size_t)r * c.W4 + w] & c.nbm[w];   // uniform
        if (!bits) continue;
        __syncwarp();
        if (lane == 0) c.todo[(size_t)r * c.W4 + w] &= ~bits;
        while (bits) {
            const int y = w * 64 + __ffsll((long long)bits) - 1;
            bits &= bits - 1ull;
            if (lane != (y & 31)) continue;
            if (y >= r) {
                // canonical bit (r, y): the candidate is open
                if (y != r) c.todo[(size_t)y * c.W4 + (r >> 6)] &= ~(1ull << (r & 63));
                k2w_certify(c, status, seg_base, r, y);
                ++got;
            } else {
                // mirror bit: confirm with the canonical one, (y, r)
                uint64_t* cw = c.todo + (size_t)y * c.W4 + (r >> 6);
                const uint64_t rb = 1ull << (r & 63);
                if (*cw & rb) {
                    *cw &= ~rb;
                    k2w_certify(c, status, seg_base, y, r);
                    ++got;
                }
            }
        }
        __syncwarp();
    }
    return got;
}

template <class Dict>
__host__ __device__ constexpr size_t k2w_dict_smem_bytes(int nb, int lds) {
    if constexpr (!Dict::IN_SMEM) return 0;
    else return (size_t)(nb > Dict::SMEM_ROW0 ? nb - Dict::SMEM_ROW0 : 0) * lds * 8;
}

// One walker = one warp.  Work item = the candidate groups (prefix, second-last row) that START in a range of `chunk`
// candidates.
template <class Dict>
__global__ void __launch_bounds__(256, 1)
k2w_walk_kernel(DevProgram P, const uint64_t* __restrict__ masks, long long n, int k_act, uint8_t* __restrict__ status,
                unsigned long long* __restrict__ queue, unsigned long long* __restrict__ counters, int chunk,
                int walker_bytes, int lds, int W4, int group_items, int split_len, uint64_t* __restrict__ witness,
                const int* __restrict__ order, long long items) {
    extern __shared__ unsigned char k2w_smem[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    constexpr int RPL = Dict::RPL;
    Dict dict;
    K2wCtx c;
    c.nb = P.wk_nb; c.nf = P.nfree; c.ld = P.wk_ld; c.lds = lds; c.R0 = P.R0; c.W4 = W4;
    c.witness = witness; c.Wm = P.W;
    {
        unsigned char* base = k2w_smem + (size_t)warp * walker_bytes;
        c.D = reinterpret_cast<double*>(base); base += k2w_dict_smem_bytes<Dict>(c.nb, lds);
        c.prow = reinterpret_cast<double*>(base); base += (size_t)Dict::PROWS * lds * 8;
        c.orig = reinterpret_cast<uint64_t*>(base); base += (size_t)c.R0 * W4 * 8;
        c.todo = reinterpret_cast<uint64_t*>(base); base += (size_t)c.R0 * W4 * 8;
        c.nbm = reinterpret_cast<uint64_t*>(base); base += (size_t)W4 * 8;
        c.bvar = reinterpret_cast<int*>(base); base += (size_t)c.nb * 4;
        c.nvar = reinterpret_cast<int*>(base); base += (size_t)c.nf * 4;
        c.where = reinterpret_cast<int*>(base); base += (size_t)c.R0 * 4;
        c.rowstart = reinterpret_cast<int*>(base); base += (size_t)c.R0 * 4;
        c.fixrow = reinterpret_cast<int*>(base);
    }
    const int W = P.W, R0 = P.R0, nb = c.nb, nf = c.nf;
    const int p = k_act >= 2 ? k_act - 2 : 0;
    unsigned long long n_piv = 0, n_give = 0, n_drop_reset = 0, n_drop_give = 0;
    int n_cert = 0;
    // prefix words / last two rows of candidate q
    auto split = [&](long long q, uint64_t (&pf)[4], int& a, int& b) {
#pragma unroll
        for (int w = 0; w < 4; ++w) pf[w] = w < W ? masks[q * W + w] : 0ull;
        b = k2w_top_bit(pf, W, &a);
        if (k_act < 2) a = b;
        pf[b >> 6] &= ~(1ull << (b & 63));
        if (k_act >= 2) pf[a >> 6] &= ~(1ull << (a & 63));
    };
    // first index in [from, limit) whose prefix (and, with a_ref >= 0, second-last row) differs from pf0 / a_ref; limit if none
    auto seg_end = [&](long long from, long long limit, const uint64_t (&pf0)[4], int a_ref) -> long long {
        for (long long q0 = from; q0 < limit; q0 += 32) {
            const long long q = q0 + lane;
            bool same = true;
            if (q < limit) {
                uint64_t m[4]; int a1, b1;
                split(q, m, a1, b1);
                same = m[0] == pf0[0] && m[1] == pf0[1] && m[2] == pf0[2] && m[3] == pf0[3] && (a_ref < 0 || a1 == a_ref);
            }
            const unsigned diff = __ballot_sync(PPG_FULL, !same);
            if (diff) return q0 + __ffs((int)diff) - 1;
        }
        return limit;
    };
    for (;;) {
        // work items are handed out most-open-candidates-first (k2w_order_items below): the cost of an item is its number
        // of open candidates, not its length, and an expensive item picked last is the tail of the launch
        unsigned long long v = 0;
        if (lane == 0) {
            v = atomicAdd(queue, 1ull);
            if (v < (unsigned long long)items && order) v = (unsigned long long)order[v];
        }
        const long long item = (long long)__shfl_sync(PPG_FULL, v, 0);
        if (item >= items) break;
        const long long c0 = item * chunk;
        const long long c1 = (c0 + chunk < n) ? c0 + chunk : n;
        // Ownership.  Work items are ranges of `chunk` candidates; a range boundary x that falls inside a prefix is moved to
        // cut(x): to the end of that prefix when less than `split` candidates of it lie beyond x (short prefixes stay whole:
        // every certificate of a vertex reaches all candidates of its prefix), else to the next (prefix, second-last row)
        // group (the first prefixes of a level own thousands of candidates: in one piece they would be the tail of the
        // launch).  Both neighbours of a boundary evaluate the same function, so the pieces tile the level.
        auto cut = [&](long long x) -> long long {
            if (x <= 0) return 0;
            if (x >= n) return n;
            uint64_t pfp[4]; int a_, b_;
            split(x - 1, pfp, a_, b_);
            const long long e = seg_end(x, n, pfp, -1);
            if (k_act < 2 || group_items == 0) return e;
            if (group_items == 2 || e - x >= (long long)split_len) return seg_end(x, n, pfp, a_);
            return e;
        };
        const long long i0 = cut(c0), own_end = cut(c1);
        long long i = i0;
        if (i >= own_end) continue;
        dict.reload(P, c, lane);
        int npiv = 0, nfixed = 0;
        bool vertex_ok = true;
        while (i < own_end) {
            // ---- segment [i, s1): candidates with the prefix of candidate i (inside what this walker owns)
            uint64_t pf0[4];
            int a0, b0;
            split(i, pf0, a0, b0);
            const long long s1 = seg_end(i + 1, own_end, pf0, -1);
            // ---- bitmaps of the segment
            for (int e = lane; e < R0 * W4; e += 32) { c.orig[e] = 0ull; c.todo[e] = 0ull; }
            __syncwarp();
            int any = 0;
            for (long long q0 = i; q0 < s1; q0 += 32) {
                const long long q = q0 + lane;
                int a1 = -1, b1 = -1;
                bool open = false;
                if (q < s1) {
                    uint64_t m[4];
                    split(q, m, a1, b1);
                    const uint8_t sb = status[q];
                    open = (sb & PPG_ST_RANK) && !(sb & PPG_ST_FEAS);
                    atomicOr(reinterpret_cast<unsigned long long*>(c.orig + (size_t)a1 * W4 + (b1 >> 6)), 1ull << (b1 & 63));
                    if ((sb & PPG_ST_RANK) && a1 != b1)
                        atomicOr(reinterpret_cast<unsigned long long*>(c.orig + (size_t)b1 * W4 + (a1 >> 6)), 1ull << (a1 & 63));
                    if (open) {
                        atomicOr(reinterpret_cast<unsigned long long*>(c.todo + (size_t)a1 * W4 + (b1 >> 6)), 1ull << (b1 & 63));
                        if (a1 != b1) atomicOr(reinterpret_cast<unsigned long long*>(c.todo + (size_t)b1 * W4 + (a1 >> 6)), 1ull << (a1 & 63));
                    }
                }
                int aprev = __shfl_up_sync(PPG_FULL, a1, 1);
                if (lane == 0) {
                    aprev = -1;
                    if (q0 > i) { uint64_t m[4]; int b2; split(q0 - 1, m, aprev, b2); }
                }
                if (q < s1 && a1 != aprev) c.rowstart[a1] = (int)(q - i);
                any |= __any_sync(PPG_FULL, open) ? 1 : 0;
            }
            __syncwarp();
            if (!any) { i = s1; continue; }
            // ---- the walk of this segment: ONE drive loop fed by a small state machine
            //   stage 0: fix prefix row f        (no marking: the prefix is not in place yet)
            //   stage 1: make row a nonbasic     (marking on)
            //   stage 2: make row b nonbasic     (marking on, a fixed as well)
            int stage = 0, f = 0, a = -1, t = -1;
            uint64_t pmask = 0ull, fm = 0ull;
            bool restart = (npiv > K2W_RESET) || !vertex_ok;
            for (;;) {
                if (restart) {
                    // (a deferring policy holds npiv mod PROWS pivots that never reached the bulk of its dictionary)
                    if (npiv % Dict::PROWS) ++(vertex_ok ? n_drop_reset : n_drop_give);
                    dict.reload(P, c, lane);
                    n_piv += npiv; npiv = 0; nfixed = 0; vertex_ok = true; restart = false;
                    stage = 0; f = 0; a = -1;
                }
                // -- next target
                if (stage == 0) {
                    if (f == 0) {
                        // keep the common head of what is fixed already
                        int keep = 0;
                        for (; keep < nfixed && keep < p; ++keep)
                            if (c.fixrow[keep] != k2w_nth(pf0, keep)) break;
                        nfixed = keep; f = keep;
                        pmask = 0ull;
                        for (int g = 0; g < nfixed; ++g) pmask |= 1ull << (~c.where[c.fixrow[g]]);
                    }
                    if (f < p) {
                        t = k2w_nth(pf0, f); fm = pmask;
                    } else {
                        n_cert += k2w_mark_all(c, status, i, lane);
                        __syncwarp();
                        if (c.witness && k_act >= 2) k2w_revisit_all(c, status, i, lane);
                        stage = 1; a = -1;
                    }
                }
                if (stage == 1) {
                    int na = -1;
                    for (int x = a + 1; x < R0 && na < 0; ++x)
                        for (int w = 0; w < W4; ++w)
                            if (c.todo[(size_t)x * W4 + w] & k2w_ge_mask(x, w)) { na = x; break; }
                    if (na < 0) break;   // segment done
                    a = na; t = a; fm = pmask;
                    if (npiv > K2W_RESET) { restart = true; continue; }   // long segment: fresh dictionary, same prefix
                }
                if (stage == 2) {
                    int b = -1;
                    for (int w = 0; w < W4 && b < 0; ++w) {
                        const uint64_t x = c.todo[(size_t)a * W4 + w] & k2w_ge_mask(a, w);
                        if (x) b = w * 64 + __ffsll((long long)x) - 1;
                    }
                    if (b < 0) { stage = 1; continue; }
                    t = b;
                }
                // -- drive row t into the nonbasic set while the columns in fm stay put
                bool reached = false;
                for (int it = 0; it < K2W_DRIVE_CAP; ++it) {
                    const int wi = c.where[t];
                    if (wi < 0) { reached = true; break; }
                    // entering column: largest positive coefficient of the target row among the free columns (degenerate
                    // target: largest magnitude - a step of length zero is feasible in either direction)
                    double bi, wbest; int j;
                    dict.target_scan(c, wi, fm, lane, bi, wbest, j);
                    const bool degen = bi <= 1e-11;
                    if (!(wbest > K2W_PIV_MIN)) break;   // s_t cannot decrease on this face (empty face / dependent row)
                    int l = wi;
                    if (!degen) {
                        // Harris ratio test over the basic rows (lanes over rows); the target row wins when it is eligible
                        double col[RPL], rat[RPL], beta[RPL];
                        double hb = CUDART_INF, trat = CUDART_INF;
                        dict.column(c, j, lane, col, beta);
#pragma unroll
                        for (int rr = 0; rr < RPL; ++rr) {
                            const int r = lane + 32 * rr;
                            const double av = col[rr];
                            col[rr] = 0.0; rat[rr] = CUDART_INF;
                            if (r < nb && av > PPG_TINY) {
                                const double bv = fmax(beta[rr], 0.0);
                                const double ia = k2w_rcp(av);
                                col[rr] = av; rat[rr] = bv * ia;
                                hb = fmin(hb, (bv + PPG_HARRIS) * ia);
                                if (r == wi) trat = rat[rr];
                            }
                        }
                        hb = warp_min_nonneg(hb);
                        trat = __shfl_sync(PPG_FULL, trat, wi & 31);
                        if (!(trat <= hb)) {
                            double lp = 0.0; int lrow = 0x7fffffff;
#pragma unroll
                            for (int rr = 0; rr < RPL; ++rr)
                                if (rat[rr] <= hb && col[rr] > lp) { lp = col[rr]; lrow = lane + 32 * rr; }
                            const double wp = warp_max_nonneg(lp);
                            l = __reduce_min_sync(PPG_FULL, (lrow != 0x7fffffff && lp == wp) ? lrow : 0x7fffffff);
                            if (l == 0x7fffffff) break;   // (cannot happen: the target row itself blocks)
                        }
                    }
                    const int rl = c.bvar[l];
                    vertex_ok = dict.pivot(c, l, j, lane);
                    ++npiv;
                    if (!vertex_ok) break;
                    if (stage != 0) {
                        n_cert += k2w_mark_row(c, status, i, rl, lane);
                        if (c.witness && k_act >= 2) k2w_revisit_row(c, status, i, rl, lane, npiv);
                    }
                    __syncwarp();
                }
                if (!vertex_ok) {
                    // a basic slack fell below the certification band: nothing is marked from such a dictionary; start over
                    // from the host vertex (this segment's open candidates stay open for the relaxation)
                    ++n_give;
                    break;
                }
                // -- what the drive means for the walk
                if (stage == 0) {
                    if (!reached) { ++n_give; break; }   // prefix not reachable here: the segment is left to the relaxation
                    if (lane == 0) c.fixrow[f] = t;
                    __syncwarp();
                    pmask |= 1ull << (~c.where[t]);
                    nfixed = ++f;
                } else if (stage == 1) {
                    if (!reached) {
                        ++n_give;
                        // nothing with this a can be certified by the walk
                        if (lane == 0) for (int w = 0; w < W4; ++w) c.todo[(size_t)a * W4 + w] &= ~k2w_ge_mask(a, w);
                        __syncwarp();
                    } else if (k_act >= 2) {
                        fm = pmask | (1ull << (~c.where[a]));
                        stage = 2;
                    }
                    // (single-row candidates were marked by the drive itself)
                } else {
                    // certified by the marking or not: this candidate is not tried again
                    if (lane == 0) c.todo[(size_t)a * W4 + (t >> 6)] &= ~(1ull << (t & 63));
                    __syncwarp();
                    if (!reached) ++n_give;
                }
            }
            i = s1;
        }
        n_piv += npiv;
    }
    n_cert = __reduce_add_sync(PPG_FULL, n_cert);
    if (lane == 0 && (n_piv || n_cert)) {
        atomicAdd(&counters[CNT_K2W_CERTIFIED], (unsigned long long)n_cert);
        atomicAdd(&counters[CNT_K2W_PIVOTS], n_piv);
        atomicAdd(&counters[CNT_K2W_WORK], n_piv * (unsigned long long)(c.nb * c.ld));
        atomicAdd(&counters[CNT_K2W_GIVEUP], n_give);
        if (n_drop_reset) atomicAdd(&counters[CNT_K2W_DROP_RESET], n_drop_reset);
        if (n_drop_give) atomicAdd(&counters[CNT_K2W_DROP_GIVEUP], n_drop_give);
    }
}

// ---- longest-processing-time-first order of the work items: cost = open candidates (rank OK, not yet certified) in the item's
// range, counting sort into K2W_COST_BUCKETS descending buckets (the order inside a bucket does not matter)
constexpr int K2W_COST_BUCKETS = 1025;

__global__ void __launch_bounds__(256) k2w_item_cost_kernel(const uint8_t* __restrict__ status, long long n, int chunk, long long items,
                                                            int* __restrict__ cost, int* __restrict__ hist) {
    const int lane = threadIdx.x & 31;
    const long long item = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (item >= items) return;
    const long long c0 = item * chunk, c1 = (c0 + chunk < n) ? c0 + chunk : n;
    int cnt = 0;
    for (long long q = c0 + lane; q < c1; q += 32) {
        const uint8_t sb = status[q];
        cnt += ((sb & PPG_ST_RANK) && !(sb & PPG_ST_FEAS)) ? 1 : 0;
    }
    cnt = __reduce_add_sync(PPG_FULL, cnt);
    if (cnt > K2W_COST_BUCKETS - 1) cnt = K2W_COST_BUCKETS - 1;
    if (lane == 0) { cost[item] = cnt; atomicAdd(&hist[K2W_COST_BUCKETS - 1 - cnt], 1); }
}

// exclusive scan of the histogram in place (one block)
__global__ void __launch_bounds__(1024) k2w_item_scan_kernel(int* __restrict__ hist) {
    __shared__ int sh[K2W_COST_BUCKETS + 1];
    for (int i = threadIdx.x; i < K2W_COST_BUCKETS; i += blockDim.x) sh[i] = hist[i];
    __syncthreads();
    if (threadIdx.x == 0) {
        int run = 0;
        for (int i = 0; i < K2W_COST_BUCKETS; ++i) { const int c = sh[i]; sh[i] = run; run += c; }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < K2W_COST_BUCKETS; i += blockDim.x) hist[i] = sh[i];
}

__global__ void __launch_bounds__(256) k2w_item_scatter_kernel(const int* __restrict__ cost, long long items, int* __restrict__ offs,
                                                               int* __restrict__ order) {
    const long long item = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (item >= items) return;
    const int pos = atomicAdd(&offs[K2W_COST_BUCKETS - 1 - cost[item]], 1);
    order[pos] = (int)item;
}

// scratch: cost (items) | order (items) | hist (K2W_COST_BUCKETS)  ints
size_t k2w_order_scratch_ints(long long n) { return (size_t)(2 * (n / 128 + 2) + K2W_COST_BUCKETS); }

static cudaError_t k2w_order_items(const uint8_t* status, long long n, int chunk, long long items, int* scratch, cudaStream_t st,
                                   const int** order_out) {
    int* cost = scratch;
    int* order = scratch + items;
    int* hist = scratch + 2 * items;
    cudaError_t e = cudaMemsetAsync(hist, 0, K2W_COST_BUCKETS * sizeof(int), st);
    if (e != cudaSuccess) return e;
    k2w_item_cost_kernel<<<(unsigned)((items * 32 + 255) / 256), 256, 0, st>>>(status, n, chunk, items, cost, hist);
    k2w_item_scan_kernel<<<1, 1024, 0, st>>>(hist);
    k2w_item_scatter_kernel<<<(unsigned)((items + 255) / 256), 256, 0, st>>>(cost, items, hist, order);
    *order_out = order;
    return cudaGetLastError();
}

#define K2W_COMMA ,
template <class Dict>
static cudaError_t launch_k2w_t(const DevProgram& P, const uint64_t* masks, long long n, int k_act, uint8_t* status,
                                unsigned long long* queue, unsigned long long* counters, int sm_count, cudaStream_t st,
                                bool* handled, uint64_t* witness, int* order_scratch) {
    const int nb = P.wk_nb, ld = P.wk_ld, lds = ld | 1, W4 = (P.R0 + 63) / 64;
    size_t wb = k2w_dict_smem_bytes<Dict>(nb, lds) + (size_t)Dict::PROWS * lds * 8 + (size_t)2 * P.R0 * W4 * 8 + (size_t)W4 * 8 +
                (size_t)(nb + P.nfree + 2 * P.R0 + K2W_MAXFIX + 2) * 4;
    wb = (wb + 15) & ~(size_t)15;
    auto kern = k2w_walk_kernel<Dict>;
    cudaFuncAttributes fa;
    cudaError_t e = cudaFuncGetAttributes(&fa, kern);
    if (e != cudaSuccess) return e;
    int wpc = (int)((size_t)(226 * 1024) / wb);
    const int by_regs = 65536 / (32 * (fa.numRegs > 0 ? fa.numRegs : 255));   // warps the register file holds
    if (wpc > by_regs) wpc = by_regs;
    if (wpc > 8) wpc = 8;
    if (wpc < 1) return cudaSuccess;   // dictionary too large for shared memory: the relaxation handles the level
    const size_t smem = wb * wpc;
    e = allow_max_smem(kern);
    if (e != cudaSuccess) return e;
    const long long walkers = (long long)sm_count * wpc;
    static const long long chunk_env = getenv("PPGPU_K2W_ITEM") ? atoll(getenv("PPGPU_K2W_ITEM")) : 0;
    // work items: small enough to balance (the first prefixes of a level own thousands of candidates each), large enough
    // to keep most groups of a prefix together (measured on levels 4-5 of the 100x30x6 program: 1024 beats 2048 and 4096)
    long long chunk = chunk_env > 0 ? chunk_env : n / (walkers * 12);
    if (chunk > 1024) chunk = 1024;
    if (chunk < 128) chunk = 128;
    long long grid = (n + chunk * wpc - 1) / (chunk * wpc);
    if (grid > sm_count) grid = sm_count;
    if (grid < 1) grid = 1;
    // ownership granularity: whole prefixes (all certificates of a vertex are used; the level is one launch and the long
    // prefixes come first in lexicographic order, so the dynamic queue schedules longest-first) or (prefix, row) groups
    // PPGPU_K2W_GROUPS: 0 whole prefixes only, 1 long prefixes are cut at group boundaries, 2 always cut at groups.
    // Default: whole prefixes while every walker has plenty of work (1 GPU, level 5 of the bench program: 60 k candidates
    // per walker; measured 236 ms whole / 243 ms cut at 2048 / 256 ms cut at 1024), cut the long ones when a walker's share
    // is small and one 6 k-candidate prefix would be the tail of the launch (a level sharded over 8 GPUs, level 4)
    static const int groups_env = getenv("PPGPU_K2W_GROUPS") ? atoi(getenv("PPGPU_K2W_GROUPS")) : -1;
    static const int split_len = getenv("PPGPU_K2W_SPLIT") ? atoi(getenv("PPGPU_K2W_SPLIT")) : 2048;
    const int group_items = groups_env >= 0 ? groups_env : (n / walkers < 16384 ? 1 : 0);
    const long long items = (n + chunk - 1) / chunk;
    const int* order = nullptr;
    static const int lpt_on = getenv("PPGPU_K2W_LPT") ? atoi(getenv("PPGPU_K2W_LPT")) : 1;
    if (lpt_on && order_scratch && items > walkers && items < (1ll << 30)) {
        if ((e = k2w_order_items(status, n, (int)chunk, items, order_scratch, st, &order)) != cudaSuccess) return e;
    }
    kern<<<(unsigned)grid, 32 * wpc, smem, st>>>(P, masks, n, k_act, status, queue, counters, (int)chunk, (int)wb, lds, W4,
                                                 group_items, split_len, witness, order, items);
    *handled = true;
    return cudaGetLastError();
}

// *handled == false: the walk is off for this program / level (no vertex dictionary, prefix too long, dictionary too large)
cudaError_t launch_k2w(const DevProgram& P, const uint64_t* masks, long long n, int k_act, uint8_t* status,
                       unsigned long long* queue, unsigned long long* counters, int sm_count, cudaStream_t st, bool* handled,
                       uint64_t* witness, int* order_scratch, bool reference) {
    *handled = false;
    static const int on = getenv("PPGPU_K2W") ? atoi(getenv("PPGPU_K2W")) : 1;
    static const int regs_on = getenv("PPGPU_K2W_REG") ? atoi(getenv("PPGPU_K2W_REG")) : 0;
    if (!on || !P.wk_ok || k_act < 1 || k_act - 2 > K2W_MAXFIX || P.W > 4 || P.nfree > 64) return cudaSuccess;
    const int rpl = (P.wk_nb + 31) / 32;
#define K2W_GO(D) return launch_k2w_t<D>(P, masks, n, k_act, status, queue, counters, sm_count, st, handled, witness, order_scratch)
    // The register-resident dictionary (instantiated for the 100 x 30 x 6 bench program: 76 basic rows x 37 columns) is
    // an EXPERIMENT, off by default (PPGPU_K2W_REG=1): 255 registers + 2 KB of spills, measured 2.6x slower per pivot than
    // the shared-memory dictionary (1395 vs 535 ms on levels 4-5); kept because it decides identically and is the
    // starting point for a leaner version
    if (regs_on && rpl == 3 && P.wk_ld == 37) K2W_GO(K2wRegDict<3 K2W_COMMA 37>);
    // (measured on levels 1..5: 317 ms against 240 ms with everything in shared memory - the register row saves 36 % of the
    // shared-memory wavefronts but pays for it with register-select code (reg_pick / reg_set jump tables, 37 selects for the
    // pivot row's owner, a serial scan of the target row): an EXPERIMENT, off by default like policy B)
    static const int hybrid_on = getenv("PPGPU_K2W_HYBRID") ? atoi(getenv("PPGPU_K2W_HYBRID")) : 0;
    if (hybrid_on && rpl == 3 && P.wk_ld == 37) K2W_GO(K2wHybridDict<3 K2W_COMMA 37>);   // the bench shape: row slot 0 in registers
    // ... everything in shared memory, columns known at compile time: updates deferred over K2W_DEFER pivots, or (the
    // reference, PPGPU_OPT_K2W_REF) every pivot applied to the whole dictionary
    if (rpl == 3 && P.wk_ld == 37 && reference) K2W_GO(K2wSmemDict<3 K2W_COMMA 37>);
    if (rpl == 3 && P.wk_ld == 37) K2W_GO(K2wDeferDict<3 K2W_COMMA 37 K2W_COMMA K2W_DEFER>);
    switch (rpl) {
        case 1: K2W_GO(K2wSmemDict<1>);
        case 2: K2W_GO(K2wSmemDict<2>);
        case 3: K2W_GO(K2wSmemDict<3>);
        case 4: K2W_GO(K2wSmemDict<4>);
        case 5: K2W_GO(K2wSmemDict<5>);
        case 6: K2W_GO(K2wSmemDict<6>);
        case 7: K2W_GO(K2wSmemDict<7>);
        case 8: K2W_GO(K2wSmemDict<8>);
        default: return cudaSuccess;
    }
#undef K2W_GO
}

}  // namespace ppgpu
