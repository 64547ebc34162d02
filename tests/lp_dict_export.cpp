// Export of the K9 start dictionary (ppopt_b200/csrc/host_math.hpp::build_lp_dictionary) for the CPU tests.  TEST
// INFRASTRUCTURE - never linked into the product; built on demand by tests/lp_dict_export.py.
#include <cstdint>
#include <cstring>

#include "../ppopt_b200/csrc/host_math.hpp"

extern "C" {

void* lpdict_create(int n, int t, int m, int q, int ne, int is_qp, const double* A, const double* b, const double* F,
                    const double* A_t, const double* b_t, const double* Q, const double* c, const double* H) {
    ppgpu::ReducedProgram* P = new ppgpu::ReducedProgram();
    if (!ppgpu::reduce_program(n, t, m, q, ne, is_qp, A, b, F, A_t, b_t, Q, c, H, *P)) { delete P; return nullptr; }
    return P;
}
void lpdict_destroy(void* h) { delete (ppgpu::ReducedProgram*)h; }

// returns lp_ok; D0 (mi x lp_ld), bvar (mi), nvar (np), obj (np x (t + 1)), X0t (n x (t + 1)) and Q2 (n x np) when ok (any
// may be null)
int lpdict_get(void* h, int* ld, double* D0, int* bvar, int* nvar, double* obj, double* X0t, double* Q2) {
    const ppgpu::ReducedProgram& P = *(const ppgpu::ReducedProgram*)h;
    *ld = P.lp_ld;
    if (!P.lp_ok) return 0;
    if (D0) std::memcpy(D0, P.lp_D0.data(), P.lp_D0.size() * sizeof(double));
    if (bvar) std::memcpy(bvar, P.lp_bvar.data(), P.lp_bvar.size() * sizeof(int));
    if (nvar) std::memcpy(nvar, P.lp_nvar.data(), P.lp_nvar.size() * sizeof(int));
    if (obj) std::memcpy(obj, P.lp_obj.data(), P.lp_obj.size() * sizeof(double));
    if (X0t) std::memcpy(X0t, P.X0t.data(), P.X0t.size() * sizeof(double));
    if (Q2) std::memcpy(Q2, P.Q2.data(), P.Q2.size() * sizeof(double));
    return 1;
}

}  // extern "C"
