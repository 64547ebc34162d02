// C export of host_math.hpp::parameter_column_maps for the CPU tests (tests/mi_maps_export.py).  TEST INFRASTRUCTURE.
#include <cstring>

#include "../ppopt_b200/csrc/host_math.hpp"

using namespace ppgpu;

extern "C" {

// Reduces the program (equality rows 0..ne-1) and writes the y maps (rows x ny) to maps, the map rows to *rows, and for an
// mpLP the dictionary's basic / nonbasic slacks (mi / np ints) and Q2 (n x np, x = x0 + Q2 v).  Returns 0, or 1 with the message in err.
int mimaps_build(int n, int t, int m, int q, int ne, int is_qp, const double* A, const double* b, const double* F,
                 const double* A_t, const double* b_t, const double* Q, const double* c, const double* H, int ny,
                 const double* Fy, const double* Hy, double* maps, int max_rows, int* rows, int* bvar, int* nvar, double* q2, char* err,
                 int errlen) {
    ReducedProgram P;
    std::string e;
    vec out;
    if (!reduce_program(n, t, m, q, ne, is_qp, A, b, F, A_t, b_t, Q, c, H, P)) e = P.error;
    else if (!parameter_column_maps(P, ny, Fy, Hy, out, e)) {}
    if (!e.empty()) { std::strncpy(err, e.c_str(), errlen - 1); err[errlen - 1] = 0; return 1; }
    *rows = parameter_map_rows(P);
    if (*rows > max_rows) { std::strncpy(err, "too many rows", errlen - 1); return 1; }
    std::memcpy(maps, out.data(), out.size() * sizeof(double));
    if (!is_qp) {
        for (int i = 0; i < P.mi; ++i) bvar[i] = P.lp_bvar[i];
        for (int j = 0; j < P.np; ++j) nvar[j] = P.lp_nvar[j];
        std::memcpy(q2, P.Q2.data(), P.Q2.size() * sizeof(double));
    }
    return 0;
}

}
