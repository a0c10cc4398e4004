// signedrank_twin.cpp -- TEST-ONLY host build of splicedice_b200/csrc/sd_signedrank_math.cuh.
// Lets the CPU test-suite check the kernel's signed-rank arithmetic against scipy and an exact
// restatement without a GPU.  Not part of the product: nothing under splicedice_b200/ loads it.
#include <stdint.h>

#include <vector>

#include "../../splicedice_b200/csrc/sd_signedrank_math.cuh"

// Per row r: n, zeros, c, 2 R+, T and the doubled ranks r2[offset[r], offset[r] + c) in, method, W, z
// (NaN unless method 2) and p out -- the kernel's per-row decisions on exact integer terms.
extern "C" void signedrank_twin_rows(int64_t rows, const int64_t *n, const int64_t *zeros, const int64_t *c,
                                     const int64_t *rp2, const int64_t *ties, const int64_t *r2, const int64_t *offset,
                                     int32_t *method, double *w, double *z, double *p)
{
    namespace sr = sd::signedrank;
    const double nan = __builtin_nan("");
    std::vector<uint64_t> counts;
    for (int64_t r = 0; r < rows; ++r) {
        method[r] = sr::method(n[r], c[r], zeros[r], ties[r]);
        const int64_t b = sr::twice_w(c[r], rp2[r]);
        w[r] = method[r] == sr::kUntested ? nan : 0.5 * (double)b;
        z[r] = method[r] == sr::kNormal ? sr::normal_z(c[r], rp2[r], ties[r]) : nan;
        if (method[r] == sr::kExact) {
            counts.assign((size_t)b + 1, 0);
            p[r] = sr::exact_p(sr::count_reference(r2 + offset[r], c[r], b, counts.data()), c[r]);
        } else {
            p[r] = method[r] == sr::kNormal ? sr::normal_p(z[r]) : nan;
        }
    }
}
