// K1 - LICQ rank screen, one warp per candidate, one lane per active row.
//
// Replaces is_full_rank(A, active_set) = (numpy.linalg.matrix_rank(A[active_set]) == |active_set|)
// (/root/reference/src/ppopt/utils/constraint_utilities.py:222-236, called from mplp_program.py:433-435).
// The program's equality rows are already projected out (host_math.hpp), so rank(A_active) = n_eq + rank of the
// k' reduced rows.  Column-pivoted Householder QR of the np x k' matrix: lane j keeps column j (= reduced row of the
// j-th active constraint) in registers, the pivot column is broadcast with shuffles, every lane reflects its own
// column.  Deficient iff |R_ss| <= PPG_RANK_TOL * |R_00|; ratios inside [PPG_RANK_BORDER_LO, PPG_RANK_BORDER_HI]
// raise PPG_ST_BORDER so that a borderline decision is never silent.
#include "common.cuh"
#include "launch.h"
#include "lp_core.cuh"

namespace ppgpu {

template <int NP, int KPL>
__global__ void __launch_bounds__(128)
k1_rank_kernel(DevProgram P, const uint64_t* __restrict__ masks, long long n, int k_act, uint8_t* __restrict__ status,
               unsigned long long* __restrict__ counters) {
    const int lane = threadIdx.x & 31;
    const long long warp0 = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
    const int W = P.W, np = P.np;
    unsigned long long n_border = 0;
    for (long long idx = warp0; idx < n; idx += nwarps) {
        const uint64_t* mk = masks + idx * W;
        uint8_t st = 0;
        const int k = k_act >= 0 ? k_act : mask_popc(mk, W);
        if (k == 0) {
            st = PPG_ST_RANK;
        } else if (k > np || k > 32 * KPL) {
            st = 0;
        } else {
            double col[KPL][NP];
            bool done[KPL];
#pragma unroll
            for (int kk = 0; kk < KPL; ++kk) {
                const int j = kk * 32 + lane;
                done[kk] = j >= k;
                const int a = (j < k) ? mask_nth(mk, W, j) : -1;
#pragma unroll
                for (int i = 0; i < NP; ++i) col[kk][i] = (a >= 0 && i < np) ? __ldg(P.At + (size_t)a * np + i) : 0.0;
            }
            double first = 0.0, minratio = 1.0;
            bool full = true;
            for (int s = 0; s < k; ++s) {
                // pivot = remaining column of largest trailing norm
                double best = -1.0; int pj = 0x7fffffff;
#pragma unroll
                for (int kk = 0; kk < KPL; ++kk) {
                    if (!done[kk]) {
                        double nn = 0.0;
#pragma unroll
                        for (int i = 0; i < NP; ++i) if (i >= s) nn = fma(col[kk][i], col[kk][i], nn);
                        if (nn > best) { best = nn; pj = kk * 32 + lane; }
                    }
                }
                warp_argmax(best, pj);
                const double rss = sqrt(best);
                if (s == 0) first = rss;
                if (first == 0.0) { full = false; minratio = 0.0; break; }
                const double ratio = rss / first;
                minratio = fmin(minratio, ratio);
                if (ratio <= PPG_RANK_TOL) { full = false; break; }
                // broadcast the pivot column, build the Householder vector v (rows s..np-1)
                double v[NP];
                const int src = pj & 31, slot = pj >> 5;
#pragma unroll
                for (int i = 0; i < NP; ++i) {
                    double x = 0.0;
#pragma unroll
                    for (int kk = 0; kk < KPL; ++kk) if (kk == slot) x = col[kk][i];
                    v[i] = (i >= s) ? shfl_d(x, src) : 0.0;
                }
                double vs = 0.0;
#pragma unroll
                for (int i = 0; i < NP; ++i) if (i == s) vs = v[i];
                const double alpha = vs >= 0.0 ? -rss : rss;
                double vtv = 0.0;
#pragma unroll
                for (int i = 0; i < NP; ++i) {
                    if (i == s) v[i] -= alpha;
                    vtv = fma(v[i], v[i], vtv);
                }
#pragma unroll
                for (int kk = 0; kk < KPL; ++kk) {
                    if (kk * 32 + lane == pj) done[kk] = true;
                    if (!done[kk] && vtv > 0.0) {
                        double d = 0.0;
#pragma unroll
                        for (int i = 0; i < NP; ++i) d = fma(v[i], col[kk][i], d);
                        d = 2.0 * d / vtv;
#pragma unroll
                        for (int i = 0; i < NP; ++i) col[kk][i] = fma(-d, v[i], col[kk][i]);
                    }
                }
            }
            if (full) st = PPG_ST_RANK;
            if (minratio > PPG_RANK_BORDER_LO && minratio < PPG_RANK_BORDER_HI) { st |= PPG_ST_BORDER; n_border++; }
        }
        if (lane == 0) status[idx] = st;
    }
    if (lane == 0) {
        if (n_border) atomicAdd(&counters[CNT_BORDER], n_border);
    }
}

template <int NP, int KPL>
static cudaError_t launch_k1_t(const DevProgram& P, const uint64_t* masks, long long n, int k_act, uint8_t* status,
                               unsigned long long* counters, int sm_count, cudaStream_t st) {
    const int threads = 128;
    long long blocks = (n * 32 + threads - 1) / threads;
    const long long cap = (long long)sm_count * 16;
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    k1_rank_kernel<NP, KPL><<<(unsigned)blocks, threads, 0, st>>>(P, masks, n, k_act, status, counters);
    return cudaGetLastError();
}



// K1p - one THREAD per candidate: unpivoted Cholesky of the k' x k' correlation block C1[act,act] in registers.
// If every Schur pivot d_j (= sin^2 of the angle between row j and the span of the rows before it) exceeds
// PPG_RANK_PRE = 1e-2, then det >= 1e-2^(k'-1), hence sigma_min^2 >= det / k'^(k'-1) >= 4.8e-21 for k' <= 8, far above
// numpy's rank threshold (sigma_max * max(k,n) * eps)^2 ~ 4e-28: the candidate is full rank, PPG_ST_RANK is set and
// the QR kernel skips it.  Everything else (2 % of the candidates, among them every truly deficient set) is handed to
// the column-pivoted QR below through PPG_ST_PRE.  The prefilter never declares a deficiency.
#define PPG_RANK_PRE 1e-2
template <int KC>
__global__ void __launch_bounds__(128)
k1_prefilter_kernel(DevProgram P, const uint64_t* __restrict__ masks, long long n, int k, uint8_t* __restrict__ status) {
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= n) return;
    const int mi = P.mi, W = P.W;
    const uint64_t* mk = masks + idx * W;
    int act[KC];
#pragma unroll
    for (int a = 0; a < KC; ++a) act[a] = (a < k) ? mask_nth(mk, W, a) : 0;
    double L[KC][KC];
#pragma unroll
    for (int a = 0; a < KC; ++a)
#pragma unroll
        for (int b = 0; b <= a; ++b) L[a][b] = (a < k && b < k) ? __ldg(P.C1 + (size_t)act[a] * mi + act[b]) : (a == b ? 1.0 : 0.0);
    bool clear = k <= P.np;
#pragma unroll
    for (int j = 0; j < KC; ++j) {
        double d = L[j][j];
#pragma unroll
        for (int c = 0; c < j; ++c) d = fma(-L[j][c], L[j][c], d);
        if (!(d > PPG_RANK_PRE)) clear = false;
        const double isd = rsqrt(d > PPG_RANK_PRE ? d : 1.0);
        L[j][j] = 1.0;
#pragma unroll
        for (int i = j + 1; i < KC; ++i) {
            double s2 = L[i][j];
#pragma unroll
            for (int c = 0; c < j; ++c) s2 = fma(-L[i][c], L[j][c], s2);
            L[i][j] = s2 * isd;
        }
    }
    status[idx] = clear ? PPG_ST_RANK : PPG_ST_PRE;
}

// Small active sets (k' <= 16): GS = 4/8/16 lanes per candidate, 32/GS candidates per warp.  Every lane of the warp
// runs the same k' Householder steps (uniform shuffles); a group that has already decided just stops updating.
template <int NP, int GS>
__global__ void __launch_bounds__(128)
k1_rank_group_kernel(DevProgram P, const uint64_t* __restrict__ masks, long long n, int k, uint8_t* __restrict__ status,
                     unsigned long long* __restrict__ counters, int use_pre) {
    constexpr int CPW = 32 / GS;
    const int lane = threadIdx.x & 31, gl = lane % GS, gid = lane / GS, gbase = gid * GS;
    const long long warp0 = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
    const int W = P.W, np = P.np;
    unsigned long long n_border = 0;
    for (long long base = warp0 * CPW; base < n; base += nwarps * CPW) {
        const long long idx = base + gid;
        bool valid = idx < n;
        if (use_pre) {
            valid = valid && (status[idx] & PPG_ST_PRE);   // cleared candidates already carry PPG_ST_RANK
            if (!__any_sync(PPG_FULL, valid)) continue;
        }
        const uint64_t* mk = masks + (valid ? idx : 0) * W;
        double col[NP];
        bool done = !(valid && gl < k);
        {
            const int a = done ? -1 : mask_nth(mk, W, gl);
#pragma unroll
            for (int i = 0; i < NP; ++i) col[i] = (a >= 0 && i < np) ? __ldg(P.At + (size_t)a * np + i) : 0.0;
        }
        double first = 0.0, minratio = 1.0;
        bool full = true, alive = valid;
        for (int s = 0; s < k; ++s) {
            double best = -1.0; int pj = gl;
            if (!done) {
                double nn = 0.0;
#pragma unroll
                for (int i = 0; i < NP; ++i) if (i >= s) nn = fma(col[i], col[i], nn);
                best = nn;
            }
#pragma unroll
            for (int o = GS / 2; o > 0; o >>= 1) {
                const double ov = shfl_xor_d(best, o);
                const int oj = __shfl_xor_sync(PPG_FULL, pj, o);
                if (ov > best || (ov == best && oj < pj)) { best = ov; pj = oj; }
            }
            const double rss = sqrt(fmax(best, 0.0));
            if (s == 0) first = rss;
            if (alive) {
                if (first == 0.0) { full = false; alive = false; minratio = 0.0; }
                else {
                    const double ratio = rss / first;
                    minratio = fmin(minratio, ratio);
                    if (ratio <= PPG_RANK_TOL) { full = false; alive = false; }
                }
            }
            double v[NP];
#pragma unroll
            for (int i = 0; i < NP; ++i) v[i] = (i >= s) ? shfl_d(col[i], gbase + pj) : 0.0;
            double vs = 0.0;
#pragma unroll
            for (int i = 0; i < NP; ++i) if (i == s) vs = v[i];
            const double alpha = vs >= 0.0 ? -rss : rss;
            double vtv = 0.0;
#pragma unroll
            for (int i = 0; i < NP; ++i) {
                if (i == s) v[i] -= alpha;
                vtv = fma(v[i], v[i], vtv);
            }
            if (gl == pj) done = true;
            if (alive && !done && vtv > 0.0) {
                double d = 0.0;
#pragma unroll
                for (int i = 0; i < NP; ++i) d = fma(v[i], col[i], d);
                d = 2.0 * d / vtv;
#pragma unroll
                for (int i = 0; i < NP; ++i) col[i] = fma(-d, v[i], col[i]);
            }
        }
        if (valid && gl == 0) {
            uint8_t st = full ? PPG_ST_RANK : 0;
            if (minratio > PPG_RANK_BORDER_LO && minratio < PPG_RANK_BORDER_HI) { st |= PPG_ST_BORDER; n_border++; }
            status[idx] = st;
        }
    }
    if (n_border) atomicAdd(&counters[CNT_BORDER], n_border);
}

template <int NP, int GS>
static cudaError_t launch_k1_g(const DevProgram& P, const uint64_t* masks, long long n, int k_act, uint8_t* status,
                               unsigned long long* counters, int sm_count, cudaStream_t st, int use_pre) {
    const int threads = 128;
    const long long per_block = (threads / 32) * (32 / GS);
    long long blocks = (n + per_block - 1) / per_block;
    const long long cap = (long long)sm_count * 16;
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    k1_rank_group_kernel<NP, GS><<<(unsigned)blocks, threads, 0, st>>>(P, masks, n, k_act, status, counters, use_pre);
    return cudaGetLastError();
}

template <int NP>
static cudaError_t launch_k1_np(const DevProgram& P, const uint64_t* masks, long long n, int k_act, uint8_t* status,
                                unsigned long long* counters, int sm_count, cudaStream_t st) {
    if (k_act >= 1 && k_act <= 8) {
        const unsigned blocks = (unsigned)((n + 127) / 128);
        if (k_act <= 2) k1_prefilter_kernel<2><<<blocks, 128, 0, st>>>(P, masks, n, k_act, status);
        else if (k_act <= 4) k1_prefilter_kernel<4><<<blocks, 128, 0, st>>>(P, masks, n, k_act, status);
        else if (k_act <= 6) k1_prefilter_kernel<6><<<blocks, 128, 0, st>>>(P, masks, n, k_act, status);
        else k1_prefilter_kernel<8><<<blocks, 128, 0, st>>>(P, masks, n, k_act, status);
        cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) return e;
        if (k_act <= 4) return launch_k1_g<NP, 4>(P, masks, n, k_act, status, counters, sm_count, st, 1);
        return launch_k1_g<NP, 8>(P, masks, n, k_act, status, counters, sm_count, st, 1);
    }
    if (k_act >= 1 && k_act <= 16) return launch_k1_g<NP, 16>(P, masks, n, k_act, status, counters, sm_count, st, 0);
    return launch_k1_t<NP, 1>(P, masks, n, k_act, status, counters, sm_count, st);
}

// Borderline escalation (SURVEY.md 7.4 item 1): candidates whose pivoted-QR ratio fell inside the borderline band are
// decided again the way the reference decides - by singular values: numpy.linalg.matrix_rank counts the singular values
// above sigma_max * max(M, N) * eps (constraint_utilities.py:236).  One warp per flagged candidate, one-sided Jacobi
// (Hestenes) on the k' x np matrix of reduced rows in shared memory: rows are rotated pairwise until mutually orthogonal,
// their norms are the singular values (small ones to high RELATIVE accuracy, which is what a rank decision at 1e-15 needs).
// Every warp scans the status bytes of the launch for PPG_ST_BORDER (70 MB at the largest level: microseconds), so no host
// round trip is needed between the QR and the feasibility stage.  The flag stays set: the decision is reported either way.
__global__ void __launch_bounds__(128)
k1_svd_recheck_kernel(DevProgram P, const uint64_t* __restrict__ masks, long long n, int k_act, uint8_t* __restrict__ status,
                      int warp_doubles) {
    extern __shared__ double k1s_smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    double* M = k1s_smem + (size_t)warp * warp_doubles;   // k x np
    const long long gw = (long long)blockIdx.x * (blockDim.x >> 5) + warp, nw = (long long)gridDim.x * (blockDim.x >> 5);
    const int W = P.W, np = P.np;
    for (long long base = gw * 32; base < n; base += nw * 32) {
        const long long mine = base + lane;
        const uint8_t sb = mine < n ? status[mine] : 0;
        unsigned todo = __ballot_sync(PPG_FULL, (sb & PPG_ST_BORDER) != 0);
        while (todo) {
            const int src = __ffs((int)todo) - 1;
            todo &= todo - 1u;
            const long long idx = base + src;
            const uint64_t* mk = masks + idx * W;
            const int k = k_act >= 0 ? k_act : mask_popc(mk, W);
            __syncwarp();
            for (int e = lane; e < k * np; e += 32) {
                const int r = e / np, c = e - r * np;
                M[e] = __ldg(P.At + (size_t)mask_nth(mk, W, r) * np + c);
            }
            __syncwarp();
            for (int sweep = 0; sweep < 40; ++sweep) {
                bool rotated = false;
                for (int p = 0; p < k - 1; ++p)
                    for (int q = p + 1; q < k; ++q) {
                        double a = 0.0, b = 0.0, g = 0.0;
                        for (int c = lane; c < np; c += 32) {
                            const double x = M[p * np + c], y = M[q * np + c];
                            a = fma(x, x, a); b = fma(y, y, b); g = fma(x, y, g);
                        }
#pragma unroll
                        for (int o = 16; o > 0; o >>= 1) { a += shfl_xor_d(a, o); b += shfl_xor_d(b, o); g += shfl_xor_d(g, o); }
                        if (fabs(g) > 1e-15 * sqrt(a * b) && g != 0.0) {
                            rotated = true;
                            const double zeta = (b - a) / (2.0 * g);
                            const double t = (zeta >= 0.0 ? 1.0 : -1.0) / (fabs(zeta) + sqrt(1.0 + zeta * zeta));
                            const double cs = 1.0 / sqrt(1.0 + t * t), sn = cs * t;
                            for (int c = lane; c < np; c += 32) {
                                const double x = M[p * np + c], y = M[q * np + c];
                                M[p * np + c] = cs * x - sn * y;
                                M[q * np + c] = sn * x + cs * y;
                            }
                        }
                        __syncwarp();
                    }
                if (!rotated) break;
            }
            double smax = 0.0, smin = CUDART_INF;
            for (int r = 0; r < k; ++r) {
                double a = 0.0;
                for (int c = lane; c < np; c += 32) a = fma(M[r * np + c], M[r * np + c], a);
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) a += shfl_xor_d(a, o);
                const double sg = sqrt(a);
                smax = fmax(smax, sg); smin = fmin(smin, sg);
            }
            // matrix_rank's tolerance, with the dimensions of the matrix the reference looks at (all active rows x n)
            const int Mr = P.ne + k, Nc = P.n;
            const double tol = smax * (double)(Mr > Nc ? Mr : Nc) * 2.220446049250313e-16;
            const bool full = k <= np && smin > tol;
            if (lane == 0) {
                const uint8_t st = status[idx];
                status[idx] = full ? (uint8_t)(st | PPG_ST_RANK) : (uint8_t)(st & ~PPG_ST_RANK);
            }
            __syncwarp();
        }
    }
}

static cudaError_t launch_k1_svd(const DevProgram& P, const uint64_t* masks, long long n, int k_act, uint8_t* status,
                                 int sm_count, cudaStream_t st) {
    const int kmax = k_act >= 0 ? k_act : P.mi;
    if (kmax < 2 || kmax > P.np) return cudaSuccess;   // one row is never borderline; more rows than columns: deficient by counting
    const int wd = kmax * P.np;
    const size_t smem = (size_t)4 * wd * sizeof(double);
    if (smem > 200 * 1024) return cudaSuccess;
    const cudaError_t e = fit_smem(k1_svd_recheck_kernel, smem);
    if (e != cudaSuccess) return e;
    long long grid = (n + 127) / 128;
    if (grid > (long long)sm_count * 4) grid = (long long)sm_count * 4;
    k1_svd_recheck_kernel<<<(unsigned)grid, 128, smem, st>>>(P, masks, n, k_act, status, wd);
    return cudaGetLastError();
}

cudaError_t launch_k1(const DevProgram& P, const uint64_t* masks, long long n, int k_act, uint8_t* status,
                      unsigned long long* counters, int sm_count, cudaStream_t st) {
    cudaError_t e = cudaErrorInvalidValue;
    if (P.np <= 8) e = launch_k1_np<8>(P, masks, n, k_act, status, counters, sm_count, st);
    else if (P.np <= 16) e = launch_k1_np<16>(P, masks, n, k_act, status, counters, sm_count, st);
    else if (P.np <= 32) e = launch_k1_np<32>(P, masks, n, k_act, status, counters, sm_count, st);
    else if (P.np <= 64) e = launch_k1_t<64, 2>(P, masks, n, k_act, status, counters, sm_count, st);
    if (e != cudaSuccess) return e;
    return launch_k1_svd(P, masks, n, k_act, status, sm_count, st);
}

}  // namespace ppgpu
