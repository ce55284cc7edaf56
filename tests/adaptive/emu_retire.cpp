// emu_retire.cpp -- TEST HELPER: host (g++) build of retire_test (csrc/sqt_paths.cuh), the function k_retire_mark
// evaluates per pixel, so that a CPU test can compare its decisions with a numpy evaluation of include/sqt.h's formula.
#include "../../squigly-trace_b200/csrc/sqt_paths.cuh"

using namespace sqt;

extern "C" {

// out[p] = 1 when pixel p (s1, s2: npix x 3) retires after n samples
void emu_retire_test(long long npix, const float *s1, const float *s2, int n, double rel_tol, double abs_tol, uint8_t *out) {
    for (long long p = 0; p < npix; ++p) out[p] = retire_test(s1 + 3 * p, s2 + 3 * p, n, rel_tol, abs_tol) ? 1 : 0;
}

}
