// Export of the K11 lifted system (ppopt_b200/csrc/host_math.hpp::build_tree_dictionary) for the CPU tests.  TEST
// INFRASTRUCTURE - never linked into the product; built on demand by tests/tree_dict_export.py.
#include <cstdint>
#include <cstring>

#include "../ppopt_b200/csrc/host_math.hpp"

extern "C" {

void* treedict_create(int n, int t, int m, int q, int ne, int nb, const int* bin, const double* A, const double* b,
                      const double* F, const double* A_t, const double* b_t, char* err, int err_len) {
    ppgpu::TreeProgram* T = new ppgpu::TreeProgram();
    if (!ppgpu::build_tree_dictionary(n, t, m, q, ne, nb, bin, A, b, F, A_t, b_t, *T)) {
        std::strncpy(err, T->error.c_str(), err_len - 1);
        err[err_len - 1] = 0;
        delete T;
        return nullptr;
    }
    return T;
}
void treedict_destroy(void* h) { delete (ppgpu::TreeProgram*)h; }

// dims: nv, rows, cols, rb0, tp, ld
void treedict_dims(void* h, int* dims) {
    const ppgpu::TreeProgram& T = *(const ppgpu::TreeProgram*)h;
    dims[0] = T.nv; dims[1] = T.rows; dims[2] = T.cols; dims[3] = T.rb0; dims[4] = T.tp; dims[5] = T.ld;
}

// D0 (rows x ld), bvar (rows), nvar (cols), hs (rows), z0 (nv), Q2 (nv x cols)
void treedict_get(void* h, double* D0, int* bvar, int* nvar, double* hs, double* z0, double* Q2) {
    const ppgpu::TreeProgram& T = *(const ppgpu::TreeProgram*)h;
    std::memcpy(D0, T.D0.data(), T.D0.size() * sizeof(double));
    std::memcpy(bvar, T.bvar.data(), T.bvar.size() * sizeof(int));
    std::memcpy(nvar, T.nvar.data(), T.nvar.size() * sizeof(int));
    std::memcpy(hs, T.hs.data(), T.hs.size() * sizeof(double));
    std::memcpy(z0, T.z0.data(), T.z0.size() * sizeof(double));
    std::memcpy(Q2, T.Q2.data(), T.Q2.size() * sizeof(double));
}

}  // extern "C"
