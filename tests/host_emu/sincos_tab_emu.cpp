// TEST-ONLY: exposes fm::sincos_tab / fm::cos_tab of option-pricing-ffn-lbfgs_b200/csrc/dhj_fastmath.cuh to ctypes.
#include "dhj_fastmath.cuh"
using namespace dhj::fm;
extern "C" {
void fm_sincos_tab(const double* x, int n, double* s, double* c) { for (int i = 0; i < n; ++i) sincos_tab(x[i], &kTables, s + i, c + i); }
void fm_cos_tab(const double* x, int n, double* c) { for (int i = 0; i < n; ++i) c[i] = cos_tab(x[i], &kTables); }
}
