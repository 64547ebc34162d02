// Fixed-theta solves of a mixed-integer program by assignment: the two small kernels around the pair mode of K8 / K9.
//
//   mi_offsets   once per assignment: its additive terms, off[a] = base + M y_a (+ 1/2 y_a' Qyy y_a on one row), where M
//                stacks the y columns of the reduced maps (host_math.hpp::parameter_column_maps), the binary-only rows
//                (b_i - A_{i,y} y), H_y' y and the linear part of the assignment's constant.  One thread per entry.
//   mi_select    after each chunk of assignments: one thread per point walks the chunk's pairs in assignment order and keeps a
//                running best, runner-up and status flags.  A pair counts when its binary-only rows hold at theta
//                (b_i + F_i theta - A_{i,y} y >= -PPG_MI_ROW_TOL (1 + |.|), |.| <= on equality rows) and its status is optimal;
//                its objective is the pass-1 value + c_y'y + 1/2 y'Qyy y + theta' H_y' y.  The minimum is strict ("<"), so among
//                exact ties the lowest assignment index wins, whatever the chunking.
#include <cmath>

#include "common.cuh"
#include "launch.h"

namespace ppgpu {

__global__ void mi_offsets_kernel(const double* __restrict__ maps, const double* __restrict__ base, int rows, int nb,
                                  const uint64_t* __restrict__ assign, long long n_assign, const double* __restrict__ qyy,
                                  int quad_row, double* __restrict__ off) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_assign * rows) return;
    const long long a = i / rows;
    const int r = (int)(i % rows);
    const uint64_t y = assign[a];
    double v = base ? base[r] : 0.0;
    for (int k = 0; k < nb; ++k)
        if ((y >> k) & 1ull) v += maps[(size_t)r * nb + k];
    if (qyy && r == quad_row) {
        double q = 0.0;
        for (int k = 0; k < nb; ++k) {
            if (!((y >> k) & 1ull)) continue;
            for (int l = 0; l < nb; ++l)
                if ((y >> l) & 1ull) q += qyy[(size_t)k * nb + l];
        }
        v += 0.5 * q;
    }
    off[i] = v;
}

__global__ void mi_select_kernel(MiSelectArgs a) {
    const long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= a.n_points) return;
    const int t = a.t, mb = a.mb;
    const double* th = a.theta + p * t;
    double best = a.best[p], second = a.second[p];
    int idx = a.best_idx[p];
    uint8_t flags = a.flags[p];
    for (int j = 0; j < a.na; ++j) {
        const long long as = a.a0 + j;
        const double* o = a.off + as * a.off_ld + a.seg;
        bool rows_hold = true;
        for (int i = 0; i < mb && rows_hold; ++i) {
            double s = o[i];
            for (int k = 0; k < t; ++k) s = fma(a.Fb[(size_t)i * t + k], th[k], s);
            const double tol = PPG_MI_ROW_TOL * (1.0 + fabs(s));
            rows_hold = a.beq[i] ? fabs(s) <= tol : s >= -tol;
        }
        if (!rows_hold) continue;
        const uint8_t st = a.pair_status[p * a.na + j];
        if (st == PPG_TLP_INFEASIBLE) continue;
        if (st == PPG_TLP_UNBOUNDED) { flags |= PPG_MI_ANY_UNBOUNDED; continue; }
        if (st != PPG_TLP_OPTIMAL) { flags |= PPG_MI_ANY_FAILED; continue; }
        double v = a.pair_obj[p * a.na + j] + o[mb + t];
        for (int k = 0; k < t; ++k) v = fma(o[mb + k], th[k], v);
        flags |= PPG_MI_ANY_OPTIMAL;
        if (v < best) { second = best; best = v; idx = (int)as; }
        else if (v < second) second = v;
    }
    a.best[p] = best; a.second[p] = second; a.best_idx[p] = idx; a.flags[p] = flags;
    a.status[p] = (flags & PPG_MI_ANY_UNBOUNDED) ? PPG_MI_UNBOUNDED : (flags & PPG_MI_ANY_FAILED) ? PPG_MI_FAILED
                : (flags & PPG_MI_ANY_OPTIMAL) ? PPG_MI_OPTIMAL : PPG_MI_INFEASIBLE;
}

cudaError_t launch_mi_offsets(const double* maps, const double* base, int rows, int nb, const uint64_t* assign, long long n_assign,
                              const double* qyy, int quad_row, double* off, cudaStream_t st) {
    const long long n = n_assign * rows;
    if (n <= 0) return cudaSuccess;
    mi_offsets_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(maps, base, rows, nb, assign, n_assign, qyy, quad_row, off);
    return cudaGetLastError();
}

cudaError_t launch_mi_select(const MiSelectArgs& a, cudaStream_t st) {
    if (a.n_points <= 0 || a.na <= 0) return cudaSuccess;
    mi_select_kernel<<<(unsigned)((a.n_points + 127) / 128), 128, 0, st>>>(a);
    return cudaGetLastError();
}

}  // namespace ppgpu
