// A dense slack dictionary held by ONE warp in shared memory, and the primal simplex rules that K9 (fixed-theta LP,
// k9_theta_lp.cu) and K11 (relaxation tree node, k11_mitree.cu) run on it.
//
// Dictionary (lp_core.cuh's convention): row r reads  x_B(r) = T[r][0] - sum_c T[r][1 + c] x_N(c).  Rows 0..m-1 are basic:
// bvar[r] >= 0 is a slack (slack r starts in row r), bvar[r] < 0 the free variable v_(-1 - bvar[r]).  Further rows (K9's
// objective row) are only carried along by the exchanges.  Columns 0..cols-1 are the nonbasic variables of the start
// dictionary (nvar), column cols is Chvatal's auxiliary x0: every slack row gets s_B = beta - D s_N + x0, the rows of v do
// not.  Variable ids: slacks 0..m-1, x0 = m.  Every slack has a tolerance tol[id] (the caller's scale); x0's is aux_tol.
//
// The rules:
//   - x0 enters on the most negative slack row below minus its tolerance (lowest row on ties);
//   - pricing over a given objective row: Dantzig (largest d_j above the optimality tolerance, lowest column on ties), or
//     Bland's rule (lowest variable id) once more than PPG_BLAND_AFTER consecutive steps were degenerate (<= PPG_DEGEN_STEP);
//   - the Harris ratio test over the slack rows only (the rows of v are free: they never block and never leave): bound
//     min (max(beta_r, 0) + tol_r) / a_r over a_r > PPG_TLP_TINY, then among the rows within the bound x0's row, else the
//     largest pivot (Bland: lowest variable id), lowest row on ties;
//   - the Gauss-Jordan exchange clamps a basic slack row whose right-hand side lands in (-tol, 0) to zero.
// A pivot splits the rows over the lanes (each lane updates its rows over all columns); pricing splits the columns, the ratio
// test the rows.  Every decision is taken on warp-reduced values, so the lanes never diverge, and depends on the dictionary
// alone, never on its batch or on the warps per CTA.
#pragma once
#include <cmath>

#include "lp_core.cuh"
#include "tolerances.h"

namespace ppgpu {

constexpr int WD_NONE = 0x7fffffff;

struct WarpDictLayout {   // per-warp scratch, in doubles
    int LD, T, P, tol, bvar, nvar, extra, stride;
};

// m basic rows, `rows` dictionary rows (m, or m + 1 with an objective row), cols nonbasic columns besides x0, and `extra`
// doubles of the caller's own after the dictionary
__host__ __device__ inline WarpDictLayout warp_dict_layout(int m, int rows, int cols, int extra) {
    WarpDictLayout o;
    o.LD = (cols + 2) | 1;   // [beta | cols | x0], odd so that lanes walking a column hit distinct banks
    int p = 0;
    o.T = p; p += rows * o.LD;
    o.P = p; p += o.LD;
    o.tol = p; p += m;
    o.bvar = p; p += (m + 1) / 2;        // ints
    o.nvar = p; p += (cols + 2) / 2;     // ints (cols + 1 columns)
    o.extra = p; p += extra;
    o.stride = p + (p & 1);              // 16-byte aligned warps
    return o;
}

struct WarpDict {
    double* T;        // rows x LD
    double* Pr;       // the pivot row (LD)
    double* tol;      // tolerance by slack id (m)
    int* bvar;        // variable of each basic row (m)
    int* nvar;        // variable of each nonbasic column (nc)
    int LD, m, rows, nc, lane;   // nc = cols + 1 columns, x0's included
    double aux_tol;   // tolerance of x0 while it is basic
    int it = 0;       // exchanges made
    int degen = 0;    // consecutive degenerate steps
    bool bland = false;

    __device__ __forceinline__ double rhs(int r) const { return T[(size_t)r * LD]; }
    __device__ __forceinline__ double tol_of(int v) const { return v == m ? aux_tol : tol[v]; }

    // one Gauss-Jordan exchange over all `rows` rows: basic row l leaves, nonbasic column j enters; false on a non-finite pivot
    __device__ __forceinline__ bool pivot(int l, int j) {
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
            if (r < m && bvar[r] >= 0 && row[0] < 0.0 && row[0] > -tol_of(bvar[r])) row[0] = 0.0;
        }
        __syncwarp();
        for (int c = lane; c <= nc; c += 32) T[(size_t)l * LD + c] = Pr[c];
        if (lane == 0) { const int b = bvar[l]; bvar[l] = nvar[j]; nvar[j] = b; }
        __syncwarp();
        ++it;
        return true;
    }

    // the row x0 enters on: the most negative slack row below minus its tolerance, WD_NONE when there is none
    __device__ __forceinline__ int x0_row() const {
        double bv = __longlong_as_double(0x7ff0000000000000ll);
        int best = WD_NONE;
        for (int r = lane; r < m; r += 32) {
            const double v = rhs(r);
            if (bvar[r] >= 0 && v < -tol[bvar[r]] && v < bv) { bv = v; best = r; }
        }
        warp_argmin(bv, best);
        return __shfl_sync(PPG_FULL, best, 0);
    }

    // the entering column for objective row orow and optimality tolerance otol, WD_NONE at the optimum.  x0's column never
    // enters: that freezes it in K9's Phase 2, and while x0 is basic no column holds it, so the test changes nothing there.
    __device__ __forceinline__ int price(const double* orow, double otol) const {
        double key = __longlong_as_double(0x7ff0000000000000ll);
        int jc = WD_NONE;
        for (int c = lane; c < nc; c += 32) {
            const double d = orow[1 + c];
            if (nvar[c] == m || !(d > otol)) continue;
            const double k = bland ? (double)nvar[c] : -d;
            if (k < key) { key = k; jc = c; }
        }
        warp_argmin(key, jc);
        return __shfl_sync(PPG_FULL, jc, 0);
    }

    struct Ratio {
        bool blocked;   // some slack row bounds the step
        int row;        // the leaving row (WD_NONE: no row within the bound, a numerical breakdown)
        double step;
    };
    // the Harris ratio test for entering column j; aux_row: x0's row (preferred among the rows within the bound), or -1
    __device__ __forceinline__ Ratio ratio(int j, int aux_row) const {
        const double INF = __longlong_as_double(0x7ff0000000000000ll);
        double hb = INF;
        for (int r = lane; r < m; r += 32) {
            if (bvar[r] < 0) continue;
            const double a = T[(size_t)r * LD + 1 + j];
            if (!(a > PPG_TLP_TINY)) continue;
            hb = fmin(hb, (fmax(rhs(r), 0.0) + tol_of(bvar[r])) / a);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) hb = fmin(hb, __shfl_xor_sync(PPG_FULL, hb, o));
        if (hb == INF) return {false, WD_NONE, INF};
        double sel = INF, step = INF;
        int lr = WD_NONE;
        for (int r = lane; r < m; r += 32) {
            if (bvar[r] < 0) continue;
            const double a = T[(size_t)r * LD + 1 + j];
            if (!(a > PPG_TLP_TINY)) continue;
            const double rat = fmax(rhs(r), 0.0) / a;
            if (!(rat <= hb)) continue;
            const double k = r == aux_row ? -INF : (bland ? (double)bvar[r] : -a);
            if (k < sel) { sel = k; lr = r; step = rat; }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const double ov = __shfl_xor_sync(PPG_FULL, sel, o);
            const int oi = __shfl_xor_sync(PPG_FULL, lr, o);
            const double os = __shfl_xor_sync(PPG_FULL, step, o);
            if (ov < sel || (ov == sel && oi < lr)) { sel = ov; lr = oi; step = os; }
        }
        return {true, __shfl_sync(PPG_FULL, lr, 0), __shfl_sync(PPG_FULL, step, 0)};
    }

    // the degenerate-step count behind Bland's rule, fed with the step of every ratio test that picked a row
    __device__ __forceinline__ void count_step(double step) {
        if (step <= PPG_DEGEN_STEP) { if (++degen > PPG_BLAND_AFTER) bland = true; } else degen = 0;
    }

    // the warp's final status: `ok` turns into PPG_TLP_NUMERIC when a basic row's right-hand side is not finite
    __device__ __forceinline__ int settle(int status, int ok) const {
        __syncwarp();
        if (status == ok)
            for (int r = lane; r < m; r += 32)
                if (!isfinite(rhs(r))) status = PPG_TLP_NUMERIC;
        return __reduce_max_sync(PPG_FULL, status);
    }

    // v into the pivot row: Pr[k] = v_k from the rows of v
    __device__ __forceinline__ void stage_v() {
        for (int r = lane; r < m; r += 32)
            if (bvar[r] < 0) Pr[-1 - bvar[r]] = rhs(r);
        __syncwarp();
    }
};

}  // namespace ppgpu
