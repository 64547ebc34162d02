// Host-side (once per program) reduction of an mpQP/mpLP to the inequality-only data the kernels read.
//
// Reference objects this replaces the per-candidate re-derivation of:
//   * equality rows are always active (reference invariant equality_indices == range(n_eq),
//     /root/reference/src/ppopt/mplp_program.py:112-118), so they are eliminated ONCE here instead of
//     inside every is_full_rank / check_feasibility / optimal_control_law call;
//   * the strictly-convex KKT system of mpqp_program.py:182-190 is rewritten through the Schur
//     complement  S = A_act Q^-1 A_act'  so a candidate only gathers a k'xk' block of a precomputed Gram.
// Pure C++ (no CUDA) so that the CPU checker in oracle/ can reuse exactly the same program reduction.
#pragma once
#include <cmath>
#include <cstdint>
#include <string>
#include <utility>
#include <vector>

namespace ppgpu {

typedef std::vector<double> vec;

struct ReducedProgram {
    // dimensions
    int n = 0, t = 0, m = 0, q = 0, ne = 0, is_qp = 0;
    int mi = 0;        // inequality rows of the main constraint body (m - ne)
    int np = 0;        // free x-directions after eliminating the equalities (n - ne)
    int W = 1;         // 64-bit words per active-set bitmask
    int R0 = 0;        // rows of the (x,theta) feasibility LP / of the theta-space region polytope: mi + q
    int nfree = 0;     // np + t free variables of the feasibility LP
    int use_gram = 0;  // 1: Q symmetric positive definite on the reduced space -> Gram/Cholesky screen
    // K1: reduced inequality rows  At (mi x np)
    vec At;
    // K2: base tableau rows (R0 x (nfree + 2)), column layout [rhs | v(np) | theta(t) | s]
    vec T0;
    // K1p: correlation matrix of the reduced rows  C1[i][j] = <At_i, At_j> / (|At_i| |At_j|)  (0 for null rows)
    vec C1;
    // K2a: Gram of the feasibility rows  Gam = Gf Gf' (R0 x R0), Gf = T0[:, 1..nfree]
    vec Gam;
    // K3: Gram G (mi x mi) and V (mi x (t+1)) with layout [const | theta coefficients]
    vec G, V;
    // K8 (fixed-theta QP, only when use_gram): x = Xp [1; theta] - K lambda  and  equality multipliers
    // mu = -Pm (Q x + H theta + c + A_in' lambda)
    vec Xp, K, Pm;   // n x (t+1), n x mi, ne x n
    // outer bounding box of Theta from the single-variable rows of A_t theta <= b_t (+-inf where there is none);
    // used by K3 as a cheap NECESSARY test: lambda_j(theta) must be able to reach >= 0 somewhere in the box
    vec th_lo, th_hi;
    // originals (row major), kept for region emission
    vec A, b, F, At_theta, bt, Q, c, H;
    // K2w: dictionary of ONE feasible vertex of {z : Gf z <= h} in slack form  s_B = beta - D s_N  (wk_nb x wk_ld,
    // column 0 = beta, column 1 + j = coefficient of the nonbasic slack wk_nvar[j]); wk_ok = 0 when the polyhedron has
    // no vertex (Gf not of full column rank), is empty, or the host phase 1 did not converge: the walk kernel is then off
    int wk_ok = 0, wk_nb = 0, wk_ld = 0;
    vec wk_D0;
    std::vector<int> wk_bvar, wk_nvar;
    // K9 (fixed-theta LP, mpLPs only): the free directions v exchanged against np inequality slacks, a dictionary whose
    // entries are constant and whose right-hand side and objective row are affine in theta.  Row i of lp_D0 (mi x lp_ld,
    // lp_ld = 1 + np + t) reads  y_i = beta0_i - D_i s_N - Dth_i theta  with layout [beta0 | D (np) | Dth (t)]; y_i is the
    // slack lp_bvar[i] >= 0, or the free variable v_c when lp_bvar[i] = -1 - c.  Column c of D is the slack lp_nvar[c].
    // Objective (the v part of (c + H theta)' x):  z = zeta - d(theta)' s_N  with lp_obj (np x (t + 1)) = [d0 | dth].
    // lp_ok = 0 when the reduced rows At have rank below np (the LP has no vertex).  x = X0t [1; theta] + Q2 v.
    int lp_ok = 0, lp_ld = 0;
    vec lp_D0, lp_obj, X0t, Q2;   // mi x lp_ld, np x (t + 1), n x (t + 1), n x np
    std::vector<int> lp_bvar, lp_nvar;
    std::string error;
};

inline bool cholesky_lower(vec& M, int n) {  // in place, lower triangle; returns false if not PD
    for (int j = 0; j < n; ++j) {
        double d = M[j * n + j];
        for (int k = 0; k < j; ++k) d -= M[j * n + k] * M[j * n + k];
        if (!(d > 0.0) || !std::isfinite(d)) return false;
        d = std::sqrt(d);
        M[j * n + j] = d;
        for (int i = j + 1; i < n; ++i) {
            double s = M[i * n + j];
            for (int k = 0; k < j; ++k) s -= M[i * n + k] * M[j * n + k];
            M[i * n + j] = s / d;
        }
    }
    return true;
}

// Householder QR of an (r x c) matrix M (row major, r >= c); returns the full orthogonal factor Qf (r x r)
// and leaves R in the upper triangle of M.
inline void householder_qr_full(vec& M, int r, int c, vec& Qf) {
    Qf.assign((size_t)r * r, 0.0);
    for (int i = 0; i < r; ++i) Qf[(size_t)i * r + i] = 1.0;
    vec v(r);
    for (int j = 0; j < c; ++j) {
        double nrm = 0.0;
        for (int i = j; i < r; ++i) nrm += M[(size_t)i * c + j] * M[(size_t)i * c + j];
        nrm = std::sqrt(nrm);
        if (nrm == 0.0) continue;
        double alpha = M[(size_t)j * c + j] >= 0 ? -nrm : nrm;
        double vtv = 0.0;
        for (int i = 0; i < r; ++i) v[i] = 0.0;
        for (int i = j; i < r; ++i) v[i] = M[(size_t)i * c + j];
        v[j] -= alpha;
        for (int i = j; i < r; ++i) vtv += v[i] * v[i];
        if (vtv == 0.0) continue;
        for (int cc = j; cc < c; ++cc) {  // M <- (I - 2vv'/v'v) M
            double d = 0.0;
            for (int i = j; i < r; ++i) d += v[i] * M[(size_t)i * c + cc];
            d = 2.0 * d / vtv;
            for (int i = j; i < r; ++i) M[(size_t)i * c + cc] -= d * v[i];
        }
        for (int rr = 0; rr < r; ++rr) {  // Qf <- Qf (I - 2vv'/v'v)
            double d = 0.0;
            for (int i = j; i < r; ++i) d += Qf[(size_t)rr * r + i] * v[i];
            d = 2.0 * d / vtv;
            for (int i = j; i < r; ++i) Qf[(size_t)rr * r + i] -= d * v[i];
        }
    }
}


// One Gauss-Jordan exchange of a slack dictionary  s_B = beta - D s_N  held as rows [beta | D] (nb x ld): basic row l
// leaves, nonbasic column j (0-based, stored in column 1 + j) enters.
inline void dict_pivot(vec& D, int nb, int ld, int l, int j) {
    const int cj = 1 + j;
    const double inv = 1.0 / D[(size_t)l * ld + cj];
    vec q(ld);
    for (int c = 0; c < ld; ++c) q[c] = D[(size_t)l * ld + c] * inv;
    q[cj] = inv;
    for (int r = 0; r < nb; ++r) {
        if (r == l) continue;
        const double col = D[(size_t)r * ld + cj];
        if (col == 0.0) continue;
        for (int c = 0; c < ld; ++c)
            if (c != cj) D[(size_t)r * ld + c] -= col * q[c];
        D[(size_t)r * ld + cj] = -col * inv;
    }
    for (int c = 0; c < ld; ++c) D[(size_t)l * ld + c] = q[c];
}

// Exchanges the free variables held in columns 0..nx-1 of a slack dictionary  s = beta - D [x; rest]  (nr x ld rows, every
// row a slack, rowvar[i] = i) against slacks, one Gauss-Jordan pivot per column on the largest remaining entry (partial
// pivoting).  Afterwards row rowvar[i] < 0 holds the free variable -1 - rowvar[i], column c < nx the slack colvar[c]; columns
// nx.. are carried along by the pivots as further right-hand sides.  Returns false when the columns have no full rank.
inline bool exchange_free_columns(vec& D, int nr, int ld, int nx, std::vector<int>& rowvar, std::vector<int>& colvar) {
    rowvar.resize(nr);
    colvar.assign(nx, -1);
    for (int i = 0; i < nr; ++i) rowvar[i] = i;
    for (int c = 0; c < nx; ++c) {
        int best = -1; double bv = 0.0;
        for (int i = 0; i < nr; ++i)
            if (rowvar[i] >= 0 && std::fabs(D[(size_t)i * ld + 1 + c]) > bv) { bv = std::fabs(D[(size_t)i * ld + 1 + c]); best = i; }
        if (best < 0 || bv < 1e-9) return false;
        dict_pivot(D, nr, ld, best, c);
        colvar[c] = rowvar[best];
        rowvar[best] = -1 - c;
    }
    return true;
}

// K2w set-up: a feasible vertex of F = {z : Gf z <= h} (Gf = T0[:, 1..nfree], h = T0[:, 0]) as a slack dictionary.
// (1) the free variables z are exchanged against slacks (exchange_free_columns; the rows that take a z are dropped: z is
// never needed again), (2) a composite phase 1 (maximise the sum of the negative slacks, Dantzig, Bland after stalling)
// makes the vertex feasible.  Runs once per program; every feasibility certificate of K2w is a vertex reached from this
// one by primal simplex pivots (k2w_walk.cu).
inline void build_walk_dictionary(ReducedProgram& P) {
    P.wk_ok = 0;
    const int R0 = P.R0, nf = P.nfree, dc = nf + 2, ld = nf + 1;
    if (nf < 1 || nf > 64 || R0 <= nf || R0 > 256) return;
    // start: every slack basic, columns = free z:  s_i = h_i - sum_c Gf[i][c] z_c
    vec D((size_t)R0 * ld);
    for (int i = 0; i < R0; ++i) {
        D[(size_t)i * ld] = P.T0[(size_t)i * dc];
        for (int c = 0; c < nf; ++c) D[(size_t)i * ld + 1 + c] = P.T0[(size_t)i * dc + 1 + c];
    }
    std::vector<int> rowvar, colvar;   // rowvar: slack id, or < 0 once the row holds a z
    if (!exchange_free_columns(D, R0, ld, nf, rowvar, colvar)) return;   // Gf has no full column rank: F has no vertex
    const int nb = R0 - nf;
    vec E((size_t)nb * ld);
    std::vector<int> bvar(nb);
    for (int i = 0, o = 0; i < R0; ++i)
        if (rowvar[i] >= 0) {
            for (int c = 0; c < ld; ++c) E[(size_t)o * ld + c] = D[(size_t)i * ld + c];
            bvar[o++] = rowvar[i];
        }
    // phase 1
    int stall = 0;
    for (int it = 0; it < 200 * (R0 + nf); ++it) {
        vec g(nf, 0.0);
        bool any = false;
        for (int i = 0; i < nb; ++i)
            if (E[(size_t)i * ld] < -1e-9) {
                any = true;
                for (int j = 0; j < nf; ++j) g[j] -= E[(size_t)i * ld + 1 + j];
            }
        if (!any) { P.wk_ok = 1; break; }
        int j = -1;
        if (stall < 20) {
            double bg = 1e-9;
            for (int c = 0; c < nf; ++c) if (g[c] > bg) { bg = g[c]; j = c; }
        } else {
            for (int c = 0; c < nf; ++c) if (g[c] > 1e-9 && (j < 0 || colvar[c] < colvar[j])) j = c;
        }
        if (j < 0) return;   // no improving direction: F is empty (or numerically so)
        auto ratio = [&](int i) {
            const double bi = E[(size_t)i * ld], a = E[(size_t)i * ld + 1 + j];
            if (bi >= -1e-9) return a > 1e-9 ? (bi > 0.0 ? bi : 0.0) / a : (double)INFINITY;   // a feasible row must stay feasible
            return a < -1e-9 ? bi / a : (double)INFINITY;                                     // an infeasible row stops at zero
        };
        double step = INFINITY;
        for (int i = 0; i < nb; ++i) step = std::fmin(step, ratio(i));
        int l = -1; double lp = 0.0;
        for (int i = 0; i < nb && step < INFINITY; ++i) {
            if (ratio(i) > step + 1e-12 * (1.0 + step)) continue;
            const double a = std::fabs(E[(size_t)i * ld + 1 + j]);
            const bool better = stall < 20 ? a > lp : (l < 0 || bvar[i] < bvar[l]);
            if (better) { l = i; lp = a; }
        }
        if (l < 0) return;
        stall = step <= 1e-12 ? stall + 1 : 0;
        dict_pivot(E, nb, ld, l, j);
        std::swap(bvar[l], colvar[j]);
    }
    if (!P.wk_ok) return;
    for (int i = 0; i < nb; ++i) if (E[(size_t)i * ld] < 0.0) E[(size_t)i * ld] = 0.0;
    for (size_t k = 0; k < E.size(); ++k) if (!std::isfinite(E[k])) { P.wk_ok = 0; return; }
    P.wk_nb = nb; P.wk_ld = ld; P.wk_D0 = E; P.wk_bvar = bvar; P.wk_nvar = colvar;
}

// K9 set-up (mpLPs): the reduced rows  s = bti + Ft theta - At v  (rows 0..mi-1 of T0, whose theta columns hold -Ft) with
// the np free directions v exchanged against slacks (exchange_free_columns, as K2w's start), and the objective row of
// (c + H theta)' x = const + g(theta)' v,  g = Q2' (c + H theta), in the nonbasic slacks.  Entries are constant, right-hand
// side and objective row affine in theta: the kernel evaluates them per point and runs the simplex from there.
inline void build_lp_dictionary(ReducedProgram& P) {
    P.lp_ok = 0;
    const int mi = P.mi, np = P.np, t = P.t, n = P.n, dc = P.nfree + 2, ld = 1 + np + t;
    vec D((size_t)mi * ld);
    for (int i = 0; i < mi; ++i)
        for (int c = 0; c < ld; ++c) D[(size_t)i * ld + c] = P.T0[(size_t)i * dc + c];
    std::vector<int> rowvar, colvar;
    if (!exchange_free_columns(D, mi, ld, np, rowvar, colvar)) return;   // At has rank below np: no vertex
    std::vector<int> vrow(np);
    for (int i = 0; i < mi; ++i) if (rowvar[i] < 0) vrow[-1 - rowvar[i]] = i;
    vec obj((size_t)np * (t + 1), 0.0);
    for (int col = 0; col <= t; ++col) {
        vec g(np);
        for (int c = 0; c < np; ++c) {
            double s = 0.0;
            for (int k = 0; k < n; ++k) s += P.Q2[(size_t)k * np + c] * (col == 0 ? P.c[k] : P.H[(size_t)k * t + col - 1]);
            g[c] = s;
        }
        for (int j = 0; j < np; ++j) {
            double s = 0.0;
            for (int c = 0; c < np; ++c) s += g[c] * D[(size_t)vrow[c] * ld + 1 + j];
            obj[(size_t)j * (t + 1) + col] = s;
        }
    }
    for (size_t k = 0; k < D.size(); ++k) if (!std::isfinite(D[k])) return;
    for (size_t k = 0; k < obj.size(); ++k) if (!std::isfinite(obj[k])) return;
    P.lp_ld = ld; P.lp_D0 = D; P.lp_obj = obj; P.lp_bvar = rowvar; P.lp_nvar = colvar;
    P.lp_ok = 1;
}

// Builds the reduced program. Inputs are row-major, equalities are rows 0..ne-1 of A/b/F.
// Q may be null for an mpLP. Returns false (and sets out.error) on malformed input.
inline bool reduce_program(int n, int t, int m, int q, int ne, int is_qp, const double* A, const double* b,
                           const double* F, const double* A_t, const double* b_t, const double* Q, const double* c,
                           const double* H, ReducedProgram& out) {
    ReducedProgram& P = out;
    P.n = n; P.t = t; P.m = m; P.q = q; P.ne = ne; P.is_qp = is_qp;
    if (n < 0 || t < 1 || m < 0 || q < 0 || ne < 0 || ne > m || ne > n) { P.error = "bad dimensions"; return false; }
    P.mi = m - ne; P.np = n - ne; P.R0 = P.mi + q; P.nfree = P.np + t;
    P.W = P.mi <= 64 ? 1 : (P.mi + 63) / 64;
    P.A.assign(A, A + (size_t)m * n); P.b.assign(b, b + m); P.F.assign(F, F + (size_t)m * t);
    P.At_theta.assign(A_t, A_t + (size_t)q * t); P.bt.assign(b_t, b_t + q);
    P.c.assign(c, c + n); P.H.assign(H, H + (size_t)n * t);
    if (is_qp) P.Q.assign(Q, Q + (size_t)n * n); else P.Q.assign((size_t)n * n, 0.0);
    const int np = P.np, mi = P.mi;
    // ---- eliminate the equalities: x = x0 + Xt*theta + Q2*v
    vec Q2((size_t)n * np, 0.0), x0(n, 0.0), Xt((size_t)n * t, 0.0), Pm((size_t)ne * n, 0.0);
    if (ne == 0) {
        for (int i = 0; i < n; ++i) Q2[(size_t)i * np + i] = 1.0;
    } else {
        vec M((size_t)n * ne), Qf;
        for (int i = 0; i < n; ++i) for (int j = 0; j < ne; ++j) M[(size_t)i * ne + j] = A[(size_t)j * n + i];
        householder_qr_full(M, n, ne, Qf);
        double rmax = 0.0;
        for (int j = 0; j < ne; ++j) rmax = std::fmax(rmax, std::fabs(M[(size_t)j * ne + j]));
        for (int j = 0; j < ne; ++j)
            if (!(std::fabs(M[(size_t)j * ne + j]) > 1e-12 * rmax)) { P.error = "equality rows are rank deficient"; return false; }
        // y1 = R^-T rhs, rhs columns = [b_eq | F_eq]; R' is lower triangular: (R')_{ij} = R_{ji}
        vec Y((size_t)ne * (t + 1));
        for (int col = 0; col <= t; ++col)
            for (int i = 0; i < ne; ++i) {
                double s = col == 0 ? b[i] : F[(size_t)i * t + col - 1];
                for (int k = 0; k < i; ++k) s -= M[(size_t)k * ne + i] * Y[(size_t)k * (t + 1) + col];
                Y[(size_t)i * (t + 1) + col] = s / M[(size_t)i * ne + i];
            }
        for (int i = 0; i < n; ++i) {
            for (int col = 0; col <= t; ++col) {
                double s = 0.0;
                for (int k = 0; k < ne; ++k) s += Qf[(size_t)i * n + k] * Y[(size_t)k * (t + 1) + col];
                if (col == 0) x0[i] = s; else Xt[(size_t)i * t + col - 1] = s;
            }
            for (int j = 0; j < np; ++j) Q2[(size_t)i * np + j] = Qf[(size_t)i * n + ne + j];
        }
        // Pm = R^-1 Q1' (A_eq' = Q1 R): the equality multipliers of a stationary point (K8)
        for (int col = 0; col < n; ++col)
            for (int i = ne - 1; i >= 0; --i) {
                double s = Qf[(size_t)col * n + i];
                for (int k = i + 1; k < ne; ++k) s -= M[(size_t)i * ne + k] * Pm[(size_t)k * n + col];
                Pm[(size_t)i * n + col] = s / M[(size_t)i * ne + i];
            }
    }
    // ---- reduced inequality rows
    P.At.assign((size_t)mi * np, 0.0);
    vec Ft((size_t)mi * t, 0.0), bti(mi, 0.0);
    for (int i = 0; i < mi; ++i) {
        const double* Ai = A + (size_t)(ne + i) * n;
        for (int j = 0; j < np; ++j) {
            double s = 0.0;
            for (int k = 0; k < n; ++k) s += Ai[k] * Q2[(size_t)k * np + j];
            P.At[(size_t)i * np + j] = s;
        }
        for (int j = 0; j < t; ++j) {
            double s = 0.0;
            for (int k = 0; k < n; ++k) s += Ai[k] * Xt[(size_t)k * t + j];
            Ft[(size_t)i * t + j] = F[(size_t)(ne + i) * t + j] - s;
        }
        double s = 0.0;
        for (int k = 0; k < n; ++k) s += Ai[k] * x0[k];
        bti[i] = b[ne + i] - s;
    }
    // ---- K2 base tableau: row = [rhs | At_i | -Ft_i | 1]  and  [bt | 0 | A_t | 1]
    const int dc = P.nfree + 2;
    P.T0.assign((size_t)P.R0 * dc, 0.0);
    for (int i = 0; i < mi; ++i) {
        double* r = &P.T0[(size_t)i * dc];
        r[0] = bti[i];
        for (int j = 0; j < np; ++j) r[1 + j] = P.At[(size_t)i * np + j];
        for (int j = 0; j < t; ++j) r[1 + np + j] = -Ft[(size_t)i * t + j];
        r[1 + np + t] = 1.0;
    }
    for (int i = 0; i < q; ++i) {
        double* r = &P.T0[(size_t)(mi + i) * dc];
        r[0] = b_t[i];
        for (int j = 0; j < t; ++j) r[1 + np + j] = A_t[(size_t)i * t + j];
        r[1 + np + t] = 1.0;
    }
    P.C1.assign((size_t)mi * mi, 0.0);
    {
        vec nr(mi, 0.0);
        for (int i = 0; i < mi; ++i) {
            double s = 0.0;
            for (int c = 0; c < np; ++c) s += P.At[(size_t)i * np + c] * P.At[(size_t)i * np + c];
            nr[i] = std::sqrt(s);
        }
        for (int i = 0; i < mi; ++i)
            for (int j = 0; j <= i; ++j) {
                double s = 0.0;
                for (int c = 0; c < np; ++c) s += P.At[(size_t)i * np + c] * P.At[(size_t)j * np + c];
                const double v = (nr[i] > 0.0 && nr[j] > 0.0) ? s / (nr[i] * nr[j]) : 0.0;
                P.C1[(size_t)i * mi + j] = P.C1[(size_t)j * mi + i] = v;
            }
    }
    P.Gam.assign((size_t)P.R0 * P.R0, 0.0);
    for (int i = 0; i < P.R0; ++i)
        for (int j = 0; j <= i; ++j) {
            double s = 0.0;
            for (int c = 0; c < P.nfree; ++c) s += P.T0[(size_t)i * dc + 1 + c] * P.T0[(size_t)j * dc + 1 + c];
            P.Gam[(size_t)i * P.R0 + j] = P.Gam[(size_t)j * P.R0 + i] = s;
        }
    P.th_lo.assign(t, -INFINITY);
    P.th_hi.assign(t, INFINITY);
    for (int i = 0; i < q; ++i) {
        int nz = 0, col = -1;
        for (int j = 0; j < t; ++j)
            if (A_t[(size_t)i * t + j] != 0.0) { ++nz; col = j; }
        if (nz == 1) {
            const double a = A_t[(size_t)i * t + col], v = b_t[i] / a;
            if (a > 0) P.th_hi[col] = std::fmin(P.th_hi[col], v); else P.th_lo[col] = std::fmax(P.th_lo[col], v);
        }
    }
    // ---- K3 Gram data (only when the reduced Hessian is symmetric positive definite)
    P.use_gram = 0;
    P.G.assign((size_t)mi * mi, 0.0);
    P.V.assign((size_t)mi * (t + 1), 0.0);
    if (is_qp) {
        double asym = 0.0, qmax = 0.0;
        for (int i = 0; i < n; ++i) for (int j = 0; j < n; ++j) {
            asym = std::fmax(asym, std::fabs(Q[(size_t)i * n + j] - Q[(size_t)j * n + i]));
            qmax = std::fmax(qmax, std::fabs(Q[(size_t)i * n + j]));
        }
        bool sym = asym <= 1e-12 * qmax;
        // Qr = Q2' Q Q2, rhs_lin = Q2'(Q [x0 | Xt] + [c | H])
        vec QQ2((size_t)n * np, 0.0), Qr((size_t)np * np, 0.0), lin((size_t)np * (t + 1), 0.0);
        for (int i = 0; i < n; ++i) for (int j = 0; j < np; ++j) {
            double s = 0.0;
            for (int k = 0; k < n; ++k) s += Q[(size_t)i * n + k] * Q2[(size_t)k * np + j];
            QQ2[(size_t)i * np + j] = s;
        }
        for (int i = 0; i < np; ++i) for (int j = 0; j < np; ++j) {
            double s = 0.0;
            for (int k = 0; k < n; ++k) s += Q2[(size_t)k * np + i] * QQ2[(size_t)k * np + j];
            Qr[(size_t)i * np + j] = s;
        }
        for (int col = 0; col <= t; ++col) {
            vec w(n);
            for (int i = 0; i < n; ++i) {
                double s = col == 0 ? c[i] : H[(size_t)i * t + col - 1];
                for (int k = 0; k < n; ++k) s += Q[(size_t)i * n + k] * (col == 0 ? x0[k] : Xt[(size_t)k * t + col - 1]);
                w[i] = s;
            }
            for (int j = 0; j < np; ++j) {
                double s = 0.0;
                for (int k = 0; k < n; ++k) s += Q2[(size_t)k * np + j] * w[k];
                lin[(size_t)j * (t + 1) + col] = s;
            }
        }
        for (int i = 0; i < np; ++i) for (int j = 0; j < i; ++j) {
            double a = 0.5 * (Qr[(size_t)i * np + j] + Qr[(size_t)j * np + i]);
            Qr[(size_t)i * np + j] = Qr[(size_t)j * np + i] = a;
        }
        vec L = Qr;
        if (sym && cholesky_lower(L, np)) {
            // Y = L^-1 At' (np x mi), Z = L^-1 lin (np x (t+1))
            vec Y((size_t)np * mi), Z((size_t)np * (t + 1));
            for (int col = 0; col < mi; ++col)
                for (int i = 0; i < np; ++i) {
                    double s = P.At[(size_t)col * np + i];
                    for (int k = 0; k < i; ++k) s -= L[(size_t)i * np + k] * Y[(size_t)k * mi + col];
                    Y[(size_t)i * mi + col] = s / L[(size_t)i * np + i];
                }
            for (int col = 0; col <= t; ++col)
                for (int i = 0; i < np; ++i) {
                    double s = lin[(size_t)i * (t + 1) + col];
                    for (int k = 0; k < i; ++k) s -= L[(size_t)i * np + k] * Z[(size_t)k * (t + 1) + col];
                    Z[(size_t)i * (t + 1) + col] = s / L[(size_t)i * np + i];
                }
            for (int i = 0; i < mi; ++i) {
                for (int j = 0; j <= i; ++j) {
                    double s = 0.0;
                    for (int k = 0; k < np; ++k) s += Y[(size_t)k * mi + i] * Y[(size_t)k * mi + j];
                    P.G[(size_t)i * mi + j] = P.G[(size_t)j * mi + i] = s;
                }
                for (int col = 0; col <= t; ++col) {
                    double s = col == 0 ? bti[i] : Ft[(size_t)i * t + col - 1];
                    for (int k = 0; k < np; ++k) s += Y[(size_t)k * mi + i] * Z[(size_t)k * (t + 1) + col];
                    P.V[(size_t)i * (t + 1) + col] = s;
                }
            }
            // K8: Qr^-1 lin = L^-T Z and Qr^-1 At' = L^-T Y, mapped back to x through Q2
            for (int col = 0; col <= t; ++col)
                for (int i = np - 1; i >= 0; --i) {
                    double s = Z[(size_t)i * (t + 1) + col];
                    for (int k = i + 1; k < np; ++k) s -= L[(size_t)k * np + i] * Z[(size_t)k * (t + 1) + col];
                    Z[(size_t)i * (t + 1) + col] = s / L[(size_t)i * np + i];
                }
            for (int col = 0; col < mi; ++col)
                for (int i = np - 1; i >= 0; --i) {
                    double s = Y[(size_t)i * mi + col];
                    for (int k = i + 1; k < np; ++k) s -= L[(size_t)k * np + i] * Y[(size_t)k * mi + col];
                    Y[(size_t)i * mi + col] = s / L[(size_t)i * np + i];
                }
            P.Xp.assign((size_t)n * (t + 1), 0.0);
            P.K.assign((size_t)n * mi, 0.0);
            for (int i = 0; i < n; ++i) {
                for (int col = 0; col <= t; ++col) {
                    double s = col == 0 ? x0[i] : Xt[(size_t)i * t + col - 1];
                    for (int k = 0; k < np; ++k) s -= Q2[(size_t)i * np + k] * Z[(size_t)k * (t + 1) + col];
                    P.Xp[(size_t)i * (t + 1) + col] = s;
                }
                for (int col = 0; col < mi; ++col) {
                    double s = 0.0;
                    for (int k = 0; k < np; ++k) s += Q2[(size_t)i * np + k] * Y[(size_t)k * mi + col];
                    P.K[(size_t)i * mi + col] = s;
                }
            }
            P.Pm = Pm;
            P.use_gram = 1;
        }
    }
    build_walk_dictionary(P);
    if (!is_qp) {
        P.X0t.assign((size_t)n * (t + 1), 0.0);
        for (int i = 0; i < n; ++i) {
            P.X0t[(size_t)i * (t + 1)] = x0[i];
            for (int j = 0; j < t; ++j) P.X0t[(size_t)i * (t + 1) + 1 + j] = Xt[(size_t)i * t + j];
        }
        P.Q2 = Q2;
        P.Pm = Pm;
        build_lp_dictionary(P);
    }
    return true;
}

// K11 (mixed-integer programs: which binary assignments have a feasible relaxation).  The LIFTED LP of a program
//   variables  z = (x, theta)  (x in program order, the binaries y = x[bin] relaxed to [l, u]),
//   rows       A x - F theta <= b (= b on the equality rows),  A_t theta <= b_t,  y_k <= u_k,  -y_k <= -l_k
// is an LP whose right-hand side is affine in the 2 nb bound values: it is reduced exactly as an mpLP whose parameters are
// p = (u_0 - 1, -l_0, u_1 - 1, -l_1, ...) (reduce_program: the equalities eliminated by QR, then build_lp_dictionary: the free
// directions v exchanged against slacks with exchange_free_columns, the bound columns carried along as right-hand sides).
// A tree node at depth d fixes y_k = v_k for k < d, i.e. p_{2k + v_k} = -1 and every other p = 0, so the right-hand side of
// dictionary row r is  beta0_r + sum_{k<d} Dbnd[r][2k + v_k]  (d loads per row), and the entries never change.
struct TreeProgram {
    int n = 0, t = 0, m = 0, q = 0, ne = 0, nb = 0;
    int nv = 0;     // n + t lifted variables
    int rows = 0;   // inequality rows of the lifted system: (m - ne) + q + 2 nb; dictionary rows (v rows included)
    int cols = 0;   // free directions v after the equalities: nv - ne
    int rb0 = 0;    // first bound row (inequality numbering): rb0 + 2k is y_k <= u_k, rb0 + 2k + 1 is -y_k <= -l_k
    int tp = 0;     // bound parameters: 2 nb (1 when nb = 0)
    int ld = 0;     // row stride of D0: 1 + cols + tp
    vec D0;         // rows x ld  [beta0 | D (cols) | Dbnd (tp)]: y_r = beta0_r - D_r s_N - Dbnd_r p
    std::vector<int> bvar, nvar;   // row r holds slack bvar[r] >= 0 or v_c for bvar[r] = -1 - c; column c is slack nvar[c]
    vec hs;         // per inequality row: 1 + |h_i| at the root bounds (u = 1, l = 0), the scale of its tolerance
    vec z0, Q2;     // z = z0 + Q2 v  (nv, nv x cols; the equality rows carry no bound parameter, so z0 is node independent)
    vec Arows, brows;  // the lifted rows, equalities first ((ne + rows) x nv) and their right-hand sides at the root bounds
    std::vector<int> bin;
    std::string error;
};

// Builds the lifted system of a program whose equality rows are rows 0..ne-1 of A / b / F.  Returns false (error set) on
// malformed input, rank-deficient equalities, or a lifted system without a vertex (rows of rank below the free variables).
inline bool build_tree_dictionary(int n, int t, int m, int q, int ne, int nb, const int* bin, const double* A,
                                  const double* b, const double* F, const double* A_t, const double* b_t, TreeProgram& T) {
    T.n = n; T.t = t; T.m = m; T.q = q; T.ne = ne; T.nb = nb;
    if (n < 1 || t < 0 || m < 0 || q < 0 || ne < 0 || ne > m || nb < 0 || nb > 63) { T.error = "bad dimensions"; return false; }
    T.bin.assign(bin, bin + nb);
    for (int k = 0; k < nb; ++k) {
        if (bin[k] < 0 || bin[k] >= n) { T.error = "binary index out of range"; return false; }
        for (int j = 0; j < k; ++j) if (bin[j] == bin[k]) { T.error = "repeated binary index"; return false; }
    }
    const int nv = n + t, tp = nb > 0 ? 2 * nb : 1, mL = m + q + 2 * nb;
    T.nv = nv; T.tp = tp;
    if (ne > nv) { T.error = "more equality rows than variables"; return false; }
    vec AL((size_t)mL * nv, 0.0), bL(mL, 0.0), FL((size_t)mL * tp, 0.0);
    for (int i = 0; i < m; ++i) {
        for (int j = 0; j < n; ++j) AL[(size_t)i * nv + j] = A[(size_t)i * n + j];
        for (int j = 0; j < t; ++j) AL[(size_t)i * nv + n + j] = -F[(size_t)i * t + j];
        bL[i] = b[i];
    }
    for (int i = 0; i < q; ++i) {
        for (int j = 0; j < t; ++j) AL[(size_t)(m + i) * nv + n + j] = A_t[(size_t)i * t + j];
        bL[m + i] = b_t[i];
    }
    for (int k = 0; k < nb; ++k) {
        const int ru = m + q + 2 * k, rl = ru + 1;
        AL[(size_t)ru * nv + bin[k]] = 1.0;  bL[ru] = 1.0; FL[(size_t)ru * tp + 2 * k] = 1.0;       // y_k <= 1 + p_2k
        AL[(size_t)rl * nv + bin[k]] = -1.0; bL[rl] = 0.0; FL[(size_t)rl * tp + 2 * k + 1] = 1.0;   // -y_k <= 0 + p_2k+1
    }
    vec c(nv, 0.0), H((size_t)nv * tp, 0.0);
    ReducedProgram R;
    if (!reduce_program(nv, tp, mL, 0, ne, 0, AL.data(), bL.data(), FL.data(), nullptr, nullptr, nullptr, c.data(), H.data(), R)) {
        T.error = R.error;
        return false;
    }
    if (!R.lp_ok) {
        T.error = "the lifted rows (program rows, Theta rows and binary bounds) have rank below the " + std::to_string(R.np) +
                  " free variables left by the equalities: the relaxation has no vertex (a continuous variable or parameter is "
                  "unbounded in some direction)";
        return false;
    }
    T.rows = R.mi; T.cols = R.np; T.rb0 = m - ne + q; T.ld = R.lp_ld;
    T.D0 = R.lp_D0; T.bvar = R.lp_bvar; T.nvar = R.lp_nvar;
    T.hs.resize(T.rows);
    for (int i = 0; i < T.rows; ++i) T.hs[i] = 1.0 + std::fabs(bL[ne + i]);
    T.z0.resize(nv);
    for (int i = 0; i < nv; ++i) T.z0[i] = R.X0t[(size_t)i * (tp + 1)];
    T.Q2 = R.Q2;
    T.Arows = AL; T.brows = bL;
    return true;
}

}  // namespace ppgpu
