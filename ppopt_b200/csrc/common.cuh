// Shared device-side declarations of libppgpu (program constants as seen by the kernels, counters, bit helpers).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "tolerances.h"

namespace ppgpu {

// Program constants resident in HBM (a few tens of KB; L1/L2 resident in practice). Built once by
// ppgpu_program_create from host_math.hpp::ReducedProgram. All matrices row-major fp64.
struct DevProgram {
    int n, t, m, q, ne, is_qp;
    int mi, np, W, R0, nfree, use_gram;
    int dc0;  // row stride of T0 = nfree + 2
    const double* At;   // mi x np      reduced inequality rows (K1)
    const double* C1;   // mi x mi      correlation matrix of the reduced rows (K1 prefilter)
    const double* T0;   // R0 x dc0     base feasibility tableau [rhs | v | theta | s] (K2)
    const double* Gam;  // R0 x R0      Gram of the feasibility rows (K2a relaxation certificates)
    const double* G;    // mi x mi      Gram  At Qr^-1 At'  (K3)
    const double* V;    // mi x (t+1)   [const | theta] right-hand sides of the Schur system (K3)
    const double* th_lo; const double* th_hi;  // t  outer bounding box of Theta (K3 multiplier-sign test)
    const double* A; const double* b; const double* F;      // originals (K5)
    const double* A_t; const double* b_t;
    const double* Q; const double* c; const double* H;
    // K8 fixed-theta QP (use_gram only): x = Xp [1; theta] - K lambda,  mu = -Pm (Q x + H theta + c + A_in' lambda)
    const double* Xp;   // n x (t+1)
    const double* K;    // n x mi
    const double* Pm;   // ne x n
    // K2a -> K2 hand-over (api.cu owns the buffers; null/0 = disabled): candidates the relaxation could not certify leave
    // the exact residuals G z* - h of their last iterate here, and the simplex starts from z* instead of the origin
    double* warm_resid;               // warm_cap x R0
    long long* warm_idx;              // warm_cap candidate indices
    unsigned long long* warm_count;   // slots handed out (may exceed warm_cap: the overflow goes the cold way)
    long long warm_cap;
    // K2w: slack dictionary of one feasible vertex of the feasibility polyhedron (host_math.hpp::build_walk_dictionary)
    int wk_ok, wk_nb, wk_ld;
    const double* wk_D0;   // wk_nb x wk_ld  [beta | D]
    const int* wk_bvar;    // wk_nb  row (slack) basic in every dictionary row
    const int* wk_nvar;    // nfree  row (slack) nonbasic in every column
    // K9 fixed-theta LP (mpLPs with a vertex only, host_math.hpp::build_lp_dictionary; Pm above is set for mpLPs too)
    int lp_ok, lp_ld;      // lp_ld = 1 + np + t
    const double* lp_D0;   // mi x lp_ld  [beta0 | D | Dth]: row = beta0 - D s_N - Dth theta
    const int* lp_bvar;    // mi          slack basic in the row, or -1 - c for the free direction v_c
    const int* lp_nvar;    // np          slack nonbasic in each column
    const double* lp_obj;  // np x (t+1)  [d0 | dth]: z = zeta - d(theta)' s_N
    const double* X0t;     // n x (t+1)   x = X0t [1; theta] + Q2 v
    const double* Q2;      // n x np
};

// Pair mode of K8 / K9 (a mixed-integer program at fixed binary assignments): work item p is the point pairs[2p] at the
// assignment pairs[2p + 1], whose additive terms are off + pairs[2p + 1] * off_ld (host_math.hpp::parameter_column_maps:
// K8 [v_y (mi) | x_y (n) | h_y (n)], K9 [d_y (mi) | f_y (mi) | x_y (n)]).  obj (may be null) receives per pair the
// continuous part of the objective, 1/2 x'Qx + (c + H theta + h_y)' x; every other output is indexed by the pair.
struct PairArgs {
    const int* pairs;
    const double* off;
    long long off_ld;
    double* obj;
};

// indices into the device counter array (uint64 each)
enum Counter {
    CNT_K1_CAND = 0,
    CNT_K2_LPS, CNT_K2_PIVOTS, CNT_K2_WORK,
    CNT_K4_LPS, CNT_K4_PIVOTS, CNT_K4_WORK,
    CNT_K5_LPS, CNT_K5_PIVOTS, CNT_K5_WORK,
    CNT_NUMERIC, CNT_BORDER, CNT_K6_LOOKUPS,          // 10, 11, 12: K6 prefix-group probes (<= k per parent)
    CNT_K2A_TRIED, CNT_K2A_CERTIFIED, CNT_K2A_STEPS,  // 13, 14, 15
    CNT_K2A_WORK,                                     // 16: steps x R0 x (1 + k') useful FMAs
    CNT_K2W_CERTIFIED, CNT_K2W_PIVOTS, CNT_K2W_WORK,  // 17, 18, 19: vertex walk (pivots x basic rows x columns FMAs)
    CNT_K2W_GIVEUP,                                   // 20: drives abandoned (iteration cap, empty face, dependent row)
    CNT_INHERITED, CNT_INHERIT_LOOKUPS,               // 21, 22: certificates inherited from parent witnesses / parents looked up
    CNT_K2W_DROP_RESET, CNT_K2W_DROP_GIVEUP,          // 23, 24: K2w reloads (K2W_RESET / vertex out of the band) that discarded
                                                      //         deferred pivots (K2wDeferDict)
    CNT_K2W_INFEASIBLE = 25,                          // 25: candidates the walk proved infeasible (drive of the last row ended at its optimum)
    CNT_K2W_INF_BAND,                                 // 26: ... drives that ended so, but whose bound fell inside PPG_WALK_INF_MARGIN's band
    CNT_COUNT = 27
};

__device__ __forceinline__ bool mask_test(const uint64_t* m, int i) { return (m[i >> 6] >> (i & 63)) & 1ull; }

__device__ __forceinline__ int mask_popc(const uint64_t* m, int W) {
    int c = 0;
    for (int w = 0; w < W; ++w) c += __popcll(m[w]);
    return c;
}

// index of the j-th (0-based) set bit, -1 if there are fewer
__device__ __forceinline__ int mask_nth(const uint64_t* m, int W, int j) {
    for (int w = 0; w < W; ++w) {
        const uint64_t x = m[w];
        const int c = __popcll(x);
        if (j < c) {
            const unsigned lo = (unsigned)x, hi = (unsigned)(x >> 32);
            const int cl = __popc(lo);
            if (j < cl) return w * 64 + (int)__fns(lo, 0, j + 1);
            return w * 64 + 32 + (int)__fns(hi, 0, j - cl + 1);
        }
        j -= c;
    }
    return -1;
}

// number of set bits strictly below position i
__device__ __forceinline__ int mask_rank(const uint64_t* m, int i) {
    int c = 0;
    const int w = i >> 6;
    for (int k = 0; k < w; ++k) c += __popcll(m[k]);
    const int b = i & 63;
    if (b) c += __popcll(m[w] & ((1ull << b) - 1ull));
    return c;
}

// highest set bit, -1 for an empty mask
__device__ __forceinline__ int mask_last(const uint64_t* m, int W) {
    for (int w = W - 1; w >= 0; --w)
        if (m[w]) return w * 64 + 63 - __clzll((long long)m[w]);
    return -1;
}

// lexicographic order of the (sorted) index lists of two equal-cardinality masks: <0, 0, >0
__device__ __forceinline__ int mask_lex_cmp(const uint64_t* a, const uint64_t* b, int W) {
    for (int w = 0; w < W; ++w) {
        const uint64_t d = a[w] ^ b[w];
        if (d) {
            const uint64_t low = d & (~d + 1ull);
            return (a[w] & low) ? -1 : 1;
        }
    }
    return 0;
}

}  // namespace ppgpu
