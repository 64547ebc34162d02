// CPU twin of the K8 fixed-theta QP kernel (ppopt_b200/csrc/k8_theta_qp.cu).  TEST INFRASTRUCTURE - never linked into the
// product; built on demand by tests/twin_theta_qp.py.  It restates the kernel's iteration sequentially on the same program
// reduction (host_math.hpp) and the same constants (tolerances.h), so that the algorithm can be checked without a GPU and the
// kernel can be compared with it decision by decision.
#include <cmath>
#include <cstdint>
#include <vector>

#include "../ppopt_b200/csrc/host_math.hpp"
#include "../ppopt_b200/csrc/tolerances.h"

using ppgpu::ReducedProgram;


// ---- K8: fixed-theta QP by a dual active-set iteration (csrc/k8_theta_qp.cu), one point at a time ----
// Same rules, tie-breaks and constants as the kernel: of the rows violated beyond their tolerance (w_r < -PPG_QP_TOL (1 +
// |w_r at lambda = 0|)) the most negative slack w_j (lowest row on ties) enters; the direction comes
// from the Cholesky factor L of G_WW (row appended on an add; on a drop the rows below shift up and the trailing block gets a
// rank-one update with the dropped column); full step to w_j = 0 or partial step to the first blocking multiplier (lowest
// row on ties), which leaves W while j stays pending.  margin: the smallest distance of any decision from its threshold or
// runner-up (slack gaps over 1 + |w|, step ratios relative), +inf when no decision had a competitor.
namespace {

inline int tri(int r, int c) { return r * (r + 1) / 2 + c; }

int theta_qp_point(const ReducedProgram& P, const double* th, double* x, double* dual, uint64_t* mask, int* iters,
                   double* margin) {
    const int mi = P.mi, np = P.np, t = P.t, t1 = t + 1, n = P.n, ne = P.ne;
    const double* G = P.G.data();
    std::vector<double> w(mi), tol(mi), lam, L((size_t)np * (np + 1) / 2), g(np), d(np), xv(np);
    std::vector<int> W;
    std::vector<char> inW(mi, 0);
    for (int r = 0; r < mi; ++r) {
        double v = P.V[(size_t)r * t1];
        for (int k = 0; k < t; ++k) v = std::fma(P.V[(size_t)r * t1 + 1 + k], th[k], v);
        w[r] = v;
        tol[r] = PPG_QP_TOL * (1.0 + std::fabs(v));
    }
    double mg = INFINITY;
    auto rel = [](double a, double b) { const double s = std::fmax(std::fabs(a), std::fabs(b)); return s > 0.0 ? std::fabs(a - b) / s : 0.0; };
    int j = -1, it = 0, status = -1;
    double lamj = 0.0;
    for (;;) {
        if (j < 0) {
            int best = -1;
            double bv = INFINITY, second = INFINITY;
            for (int r = 0; r < mi; ++r) {
                if (inW[r]) continue;
                mg = std::fmin(mg, std::fabs(w[r] + tol[r]) / (1.0 + std::fabs(w[r])));
                if (!(w[r] < -tol[r])) continue;
                if (w[r] < bv) { second = bv; bv = w[r]; best = r; }
                else if (w[r] < second) second = w[r];
            }
            if (best < 0) { status = PPG_QP_OPTIMAL; break; }
            if (second < INFINITY) mg = std::fmin(mg, (second - bv) / (1.0 + std::fabs(bv)));
            j = best;
            lamj = 0.0;
        }
        if (it >= PPG_QP_MAX_ITER) { status = PPG_QP_ITERLIM; break; }
        ++it;
        const int nW = (int)W.size();
        for (int i = 0; i < nW; ++i) g[i] = G[(size_t)W[i] * mi + j];
        for (int i = 0; i < nW; ++i) {
            const double gi = g[i] / L[tri(i, i)];
            g[i] = gi;
            for (int r = i + 1; r < nW; ++r) g[r] = std::fma(-L[tri(r, i)], gi, g[r]);
        }
        double ll = 0.0;
        for (int i = 0; i < nW; ++i) ll = std::fma(g[i], g[i], ll);
        const double gjj = G[(size_t)j * mi + j], z = gjj - ll;
        for (int i = 0; i < nW; ++i) d[i] = -g[i];
        for (int i = nW - 1; i >= 0; --i) {
            const double di = d[i] / L[tri(i, i)];
            d[i] = di;
            for (int r = 0; r < i; ++r) d[r] = std::fma(-L[tri(i, r)], di, d[r]);
        }
        mg = std::fmin(mg, gjj > 0.0 ? std::fabs(z - PPG_QP_CURV * gjj) / gjj : 0.0);
        const bool full = z > PPG_QP_CURV * gjj;
        const double sf = full ? -w[j] / z : INFINITY;
        int p = -1;
        double sb = INFINITY, sb2 = INFINITY;
        for (int i = 0; i < nW; ++i) {
            if (!(d[i] < -PPG_QP_DTOL)) continue;
            const double rt = lam[i] / -d[i];
            if (rt < sb || (rt == sb && W[i] < W[p])) { sb2 = sb; sb = rt; p = i; }
            else if (rt < sb2) sb2 = rt;
        }
        if (sb2 < INFINITY) mg = std::fmin(mg, rel(sb, sb2));
        if (sb < INFINITY && sf < INFINITY) mg = std::fmin(mg, rel(sb, sf));
        if (p < 0 && !full) { status = PPG_QP_INFEASIBLE; break; }
        const bool partial = sb < sf;
        const double s = partial ? sb : sf;
        if (!std::isfinite(s)) { status = PPG_QP_NUMERIC; break; }
        for (int r = 0; r < mi; ++r) {
            double u = G[(size_t)j * mi + r];
            for (int k = 0; k < nW; ++k) u = std::fma(G[(size_t)W[k] * mi + r], d[k], u);
            w[r] = std::fma(s, u, w[r]);
        }
        for (int k = 0; k < nW; ++k) lam[k] = std::fma(s, d[k], lam[k]);
        lamj += s;
        if (partial) {
            // drop position p: rows below shift up without column p, trailing block += x x' (x = old column p below p)
            for (int r = p + 1; r < nW; ++r) xv[r - 1] = L[tri(r, p)];
            for (int r = p + 1; r < nW; ++r)
                for (int c = 0; c <= r; ++c)
                    if (c != p) L[tri(r - 1, c - (c > p))] = L[tri(r, c)];
            bool ok = true;
            for (int k = p; k < nW - 1; ++k) {
                const double lkk = L[tri(k, k)], xk = xv[k];
                const double rr = std::sqrt(std::fma(lkk, lkk, xk * xk)), c = rr / lkk, sn = xk / lkk;
                for (int i = k + 1; i < nW - 1; ++i) {
                    const double lik = (L[tri(i, k)] + sn * xv[i]) / c;
                    L[tri(i, k)] = lik;
                    xv[i] = c * xv[i] - sn * lik;
                }
                L[tri(k, k)] = rr;
                ok = ok && rr > 0.0 && std::isfinite(rr);
            }
            inW[W[p]] = 0;
            W.erase(W.begin() + p);
            lam.erase(lam.begin() + p);
            if (!ok) { status = PPG_QP_NUMERIC; break; }
        } else {
            if (nW >= np) { status = PPG_QP_NUMERIC; break; }
            for (int i = 0; i < nW; ++i) L[tri(nW, i)] = g[i];
            L[tri(nW, nW)] = std::sqrt(z);
            W.push_back(j);
            lam.push_back(lamj);
            inW[j] = 1;
            j = -1;
        }
    }
    for (int wd = 0; wd < P.W; ++wd) mask[wd] = 0;
    for (int r : W) mask[r >> 6] |= 1ull << (r & 63);
    *iters = it;
    *margin = mg;
    const int nW = (int)W.size();
    if (status != PPG_QP_OPTIMAL) {
        if (x) for (int i = 0; i < n; ++i) x[i] = NAN;
        if (dual) for (int i = 0; i < P.m; ++i) dual[i] = NAN;
        return status;
    }
    std::vector<double> xl(n), res(n);
    for (int i = 0; i < n; ++i) {
        double v = P.Xp[(size_t)i * t1];
        for (int k = 0; k < t; ++k) v = std::fma(P.Xp[(size_t)i * t1 + 1 + k], th[k], v);
        for (int k = 0; k < nW; ++k) v = std::fma(-P.K[(size_t)i * mi + W[k]], lam[k], v);
        xl[i] = v;
    }
    for (int i = 0; i < n; ++i) {
        double v = P.c[i];
        for (int k = 0; k < t; ++k) v = std::fma(P.H[(size_t)i * t + k], th[k], v);
        for (int k = 0; k < n; ++k) v = std::fma(P.Q[(size_t)i * n + k], xl[k], v);
        for (int k = 0; k < nW; ++k) v = std::fma(P.A[(size_t)(ne + W[k]) * n + i], lam[k], v);
        res[i] = v;
    }
    if (x) for (int i = 0; i < n; ++i) x[i] = xl[i];
    if (dual) {
        for (int e = 0; e < ne; ++e) {
            double v = 0.0;
            for (int i = 0; i < n; ++i) v = std::fma(P.Pm[(size_t)e * n + i], res[i], v);
            dual[e] = -v;
        }
        for (int r = 0; r < mi; ++r) dual[ne + r] = 0.0;
        for (int k = 0; k < nW; ++k) dual[ne + W[k]] = lam[k];
    }
    return status;
}

}  // namespace

extern "C" {

void* k8twin_create(int n, int t, int m, int q, int ne, int is_qp, const double* A, const double* b, const double* F,
                    const double* A_t, const double* b_t, const double* Q, const double* c, const double* H) {
    ReducedProgram* P = new ReducedProgram();
    if (!ppgpu::reduce_program(n, t, m, q, ne, is_qp, A, b, F, A_t, b_t, Q, c, H, *P)) { delete P; return nullptr; }
    return P;
}
void k8twin_destroy(void* h) { delete (ReducedProgram*)h; }
int k8twin_words(void* h) { return ((ReducedProgram*)h)->W; }
int k8twin_use_gram(void* h) { return ((ReducedProgram*)h)->use_gram; }

// n points (theta n x t): status, x (n x num_x), dual (n x m), working-set masks (n x W), iterations, decision margins;
// returns -2 when the program has no Gram data (mpLP, or a reduced Hessian that is not positive definite)
int k8twin_theta_qp(void* h, const double* theta, long npts, uint8_t* status, double* x, double* dual, uint64_t* mask,
                    int32_t* iters, double* margin) {
    const ReducedProgram& P = *(const ReducedProgram*)h;
    if (!P.is_qp || !P.use_gram) return -2;
    for (long i = 0; i < npts; ++i) {
        int it = 0;
        double mg = 0.0;
        status[i] = (uint8_t)theta_qp_point(P, theta + i * P.t, x + i * P.n, dual + i * P.m, mask + i * P.W, &it, &mg);
        iters[i] = it;
        margin[i] = mg;
    }
    return 0;
}

}  // extern "C"
