// TEST-ONLY host build of torchflows_b200/csrc/b2f_rqfast.cuh (g++, -ffp-contract=off) for
// tests/test_tcq_specialise_host.py: the polynomial knot derivative and the output-only inverse map.
#include "../torchflows_b200/csrc/b2f_math.cuh"
#include "../torchflows_b200/csrc/b2f_rqfast.cuh"

using namespace b2f;

extern "C" {
// delta at the logits kRqEdgeU + u
void ts_delta_poly(const float* u, float* out, int64_t n) {
    for (int64_t i = 0; i + 1 < n; i += 2) {
        const f2 d = rqf::delta_poly(mk2(u[i], u[i + 1]));
        out[i] = d.x;
        out[i + 1] = d.y;
    }
    if (n & 1) out[n - 1] = rqf::delta_poly(mk2(u[n - 1], u[n - 1])).x;
}

float ts_edge_u() { return kRqEdgeU; }
float ts_delta_poly_bound() { return rqf::kDeltaPolyBound; }

// fast-variant inverse map on the 24 folded columns per element: out and log2-det (NaN where LD = 0 leaves it unwritten)
void ts_inverse(const float* x, const float* g, float* out, float* ld2, int64_t n, float b, int dpoly, int ld) {
    for (int64_t i = 0; i < n; ++i) {
        float gg[24];
        for (int j = 0; j < 24; ++j) gg[j] = g[i * 24 + j];
        float l = __builtin_nanf("");
        if (dpoly && ld) rqf::inverse<false, 0, true, true>(x[i], gg, b, out[i], l);
        else if (dpoly) rqf::inverse<false, 0, true, false>(x[i], gg, b, out[i], l);
        else if (ld) rqf::inverse<false, 0, false, true>(x[i], gg, b, out[i], l);
        else rqf::inverse<false, 0, false, false>(x[i], gg, b, out[i], l);
        ld2[i] = l;
    }
}
}
