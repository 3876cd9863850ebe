// Rational-quadratic spline transformer, "folded" formulation for the tensor-core coupling kernel
// (b2f_flow_tcq.cu).  Same function as rq_apply in b2f_math.cuh (reference: transformers/spline/base.py:29-72,
// transformers/spline/rational_quadratic.py:45-200), restructured so that one element costs ~150 issue slots
// instead of ~540:
//
//  * the output layer of the conditioner is linear, so every *linear* step of the parameterisation is folded into
//    its weights when the operands are laid out (torchflows_b200/_tcq.py): the 24 GEMM columns of an element are
//        g[0..8)   L_j  = log2(e) * u_x[j]                      widths logits, ready for ex2
//        g[8..16)  Dl_j = log2(e) * u_y[j] / 1000               heights logits are L_j + Dl_j  (rational_quadratic.py:76)
//        g[16..24) Dd_i = a[i+1] - a[i],  a = c + [c, u_d, c]/1000   differences of the padded derivative logits
//    (rational_quadratic.py:77,125-127: the pad value c is itself divided by 1000), so a[k] and a[k+1] are prefix sums
//    selected by the search predicates;
//  * knots are never materialised: the search runs on the normalised cumulative bin sizes against
//    t = (v + b) / 2b, and the quantities of the selected bin (lower knot, upper knot for x and y, the two
//    derivative logits) are accumulated with *predicated adds* under the 7 search predicates (monotone, so the
//    predicated prefix sum IS the k-th cumulative sum, in the reference's summation order);
//  * heights softmax: exp(L + Dl) = exp(L) * 2^Dl with a cubic for 2^Dl when the host proves |Dl| < 1/32 from the
//    weights (|tanh| <= 1), else the SFU;  no max-subtraction when the host proves |L| < 40 (same bound);
//  * one reciprocal for both softmax normalisations, one for the rational function (everything multiplied through by
//    w^3), one lg2 for the log-determinant;  the log-det is returned in log2 units and scaled once per row;
//  * knot derivatives: a cubic for softplus when the host proves |a - c| < 1/32 from the weights (DPOLY), else the SFU;
//  * the inverse map can skip its log-determinant altogether (LD = false: Flow.sample without log_prob); the output chain
//    never reads the log-det arithmetic, so `out` is bit-identical either way.
//
// Tolerance-checked (1e-4 abs/rel on log_prob), not bit-checked: the bit-exact bin index contract belongs to the
// stand-alone transformer kernel (b2f_math.cuh), whose parameters are fp32-faithful; here they come out of a TF32 GEMM.
#pragma once
#include "b2f_math.cuh"

namespace b2f {
namespace rqf {

constexpr float kLog2e = 1.4426950408889634f;
constexpr float kLn2 = 0.6931471805599453f;
constexpr float kSizeScale = 0.992f;          // 1 - 1e-3 * 8   (rational_quadratic.py:47, n_bins = 8)
constexpr float kPolyBound = 1.0f / 32.0f;    // |Dl| below which the cubic 2^Dl is exact to 1e-8
constexpr float kNoMaxBound = 40.0f;          // |L| below which ex2 needs no max subtraction
constexpr float kEdgeLogit = kRqEdgeU + kRqEdgeU / 1000.0f;   // logit of the two padded edge derivatives: c + c/1000
// |a - c| (derivative logit a, c = kRqEdgeU) below which delta_poly is within 1 ulp of the exact delta: the cubic's
// truncation error is < 4e-9 there, the rest is the rounding of the last FMA (tests/test_tcq_specialise_host.py)
constexpr float kDeltaPolyBound = 1.0f / 32.0f;

B2F_HD float f_ex2(float x) {
#if defined(__CUDA_ARCH__)
    float y; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y;
#else
    return exp2f(x);
#endif
}
B2F_HD float f_lg2(float x) {
#if defined(__CUDA_ARCH__)
    float y; asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y;
#else
    return log2f(x);
#endif
}
B2F_HD float f_rcp(float x) {
#if defined(__CUDA_ARCH__)
    float y; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y;
#else
    return 1.0f / x;
#endif
}
B2F_HD float f_sqrt(float x) {
#if defined(__CUDA_ARCH__)
    float y; asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y;
#else
    return sqrtf(x);
#endif
}

// derivative at a knot from its logit: 1e-5 + softplus(a)   (rational_quadratic.py:77)
B2F_HD float delta(float a) {
    const float e = f_ex2(fminf(a, 80.0f) * kLog2e);
    return fmaf(f_lg2(1.0f + e), kLn2, kRqMinDelta);
}

// delta at the two knot logits kRqEdgeU + u.x, kRqEdgeU + u.y for |u| < kDeltaPolyBound: Taylor cubic of 1e-5 + softplus
// around c = kRqEdgeU, coefficients in fp64 at the fp32 value of c.  softplus(c) = 1 - 1e-5 (rational_quadratic.py:38), so
// the constant term is 1 (1 + 1.5e-8 in fp64).  The first step is two scalar FMAs: they take both coefficients as
// immediates, where FFMA2 would hold its multiplier in a register across the chunk loop (+2 registers in the sampling kernel).
B2F_HD f2 delta_poly(f2 u) {
    f2 p = mk2(fmaf(u.x, -0.01024104604576881f, 0.1162725642742006f), fmaf(u.y, -0.01024104604576881f, 0.1162725642742006f));
    p = pk_fma(p, u, mk2(0.6321168855657702f, 0.6321168855657702f));
    return pk_fma(p, u, mk2(1.0f, 1.0f));
}

struct Sel {            // the selected bin: knots measured from -b (cumulative bin sizes in [0, 2b]), derivative logits
    float xl, xu, yl, yu, dl0, dl1;     // DPOLY: dl0, dl1 are the logits minus kRqEdgeU
};

template <bool DPOLY>
B2F_HD f2 knot_deltas(const Sel& s) {
    return DPOLY ? delta_poly(mk2(s.dl0, s.dl1)) : mk2(delta(s.dl0), delta(s.dl1));
}

// One search step with the predicate as a number, m = (c < t) ? 1 : 0:  lo += m a, up += m b (packed pairs),
// dl0 += m d0, dl1 += m d1.  fma(1, x, acc) rounds exactly like acc + x, so this IS the predicated sum; as FFMA2 / FFMA
// it stays on the FMA pipe (ptxas turns predicated packed adds into 32-bit selects on the half-rate ALU pipe).
B2F_HD float select_step(float c, float t, f2& lo, f2& up, float& dl0, float& dl1, f2 a, f2 b, float d0, float d1) {
    const float m = c < t ? 1.0f : 0.0f;
    const f2 mm = mk2(m, m);
    lo = pk_fma(mm, a, lo);
    up = pk_fma(mm, b, up);
    dl0 = fmaf(m, d0, dl0);
    dl1 = fmaf(m, d1, dl1);
    return m;
}

// Softmaxes, search and selection.  t = v + b.  INV: search on the y knots (rational_quadratic.py:147).
// SAFE: max-subtracted exponentials and SFU for the heights (no host-side bound on the logits).
// NY (even): how many of the 8 heights exponentials go to the SFU in the fast variant (pipe balancing; any value is exact).
// DPOLY: derivative logits accumulated relative to kRqEdgeU (the offsets delta_poly takes).
// Widths and heights travel as packed pairs (.x widths, .y heights): FADD2 / FFMA2 issue once for both.
template <bool INV, bool SAFE, int NY, bool DPOLY = false>
B2F_HD void select(const float (&g)[24], float t, float two_b, Sel& s) {
    static_assert(NY % 2 == 0, "the cubic 2^d is evaluated on pairs of logits");
    f2 e[8];
    float m = 0.0f;
    if (SAFE) {
        m = g[0];
#pragma unroll
        for (int j = 1; j < 8; ++j) m = fmaxf(m, g[j]);
    }
#pragma unroll
    for (int j = 0; j < 8; j += 2) {
        const float a0 = SAFE ? g[j] - m : g[j], a1 = SAFE ? g[j + 1] - m : g[j + 1];
        e[j].x = f_ex2(a0);
        e[j + 1].x = f_ex2(a1);
        if (SAFE || j < NY) {
            e[j].y = f_ex2(a0 + g[8 + j]);
            e[j + 1].y = f_ex2(a1 + g[9 + j]);
        } else {                               // 2^d, |d| < 1/32: 1 + d ln2 + (d ln2)^2/2 + (d ln2)^3/6, two logits at a time
            const f2 d = mk2(g[8 + j], g[9 + j]);
            f2 p = pk_fma(d, mk2(0.0555041086648216f, 0.0555041086648216f), mk2(0.2402265069591007f, 0.2402265069591007f));
            p = pk_fma(p, d, mk2(kLn2, kLn2));
            p = pk_fma(p, d, mk2(1.0f, 1.0f));
            e[j].y = e[j].x * p.x;
            e[j + 1].y = e[j + 1].x * p.y;
        }
    }
    const f2 sum = pk_add(pk_add(pk_add(e[0], e[1]), pk_add(e[2], e[3])), pk_add(pk_add(e[4], e[5]), pk_add(e[6], e[7])));
    const float r = (kSizeScale * two_b) * f_rcp(sum.x * sum.y);
    const f2 rr = mk2(r * sum.y, r * sum.x);
    // bin sizes in units of the spline range: 2b (1e-3 + 0.992 softmax)   (rational_quadratic.py:46-49)
    const float minb = kRqMinBin * two_b;
    f2 sz[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) sz[j] = pk_fma(e[j], rr, mk2(minb, minb));
    f2 lo = mk2(0.0f, 0.0f), up = sz[0];
    const float edge = DPOLY ? kRqEdgeU / 1000.0f : kEdgeLogit;
    s.dl0 = edge; s.dl1 = edge + g[16];
    float c = 0.0f, m7 = 0.0f;
#pragma unroll
    for (int j = 1; j < 8; ++j) {
        c += INV ? sz[j - 1].y : sz[j - 1].x;             // cumulative size = knot j in normalised units
        // searchsorted(right=False): knots strictly below v are counted
        m7 = select_step(c, t, lo, up, s.dl0, s.dl1, sz[j - 1], sz[j], g[16 + j - 1], g[16 + j]);
    }
    if (m7 != 0.0f) up = mk2(two_b, two_b);               // bins[K] = +b is pinned (rational_quadratic.py:52)
    s.xl = lo.x; s.yl = lo.y; s.xu = up.x; s.yu = up.y;
}

// Forward map (rational_quadratic.py:88-109, log-det :56-63).  out = spline(v), ld2 = log2 |d out / d v|.
template <bool SAFE, int NY, bool DPOLY = false>
B2F_HD void forward(float v, const float (&g)[24], float b, float& out, float& ld2) {
    const float two_b = b + b;
    const bool inb = fabsf(v) < b;                        // strict, spline/base.py:29-33; NaN -> identity tail
    const float t = v + b;
    Sel s;
    select<false, SAFE, NY, DPOLY>(g, t, two_b, s);
    const float w = s.xu - s.xl, hgt = s.yu - s.yl;
    const float yk = s.yl - b;
    const float a = fminf(fmaxf(t - s.xl, 0.0f), w);      // v - x_k = xi * w, xi clipped to [0, 1]  (:99)
    const f2 dd = knot_deltas<DPOLY>(s);
    const float d0 = dd.x, d1 = dd.y;
    // out = yk + hgt (s xi^2 + d0 q) / (s + t1 q), everything multiplied through by w^3:
    const float wa = w - a, aw = a * wa, h2 = hgt + hgt;
    const float T = fmaf(w, d0 + d1, -h2);                // w * t1
    const float den = fmaf(T, aw, (hgt * w) * w);         // w^3 (s + t1 q)
    const float num = fmaf(hgt * a, a, (w * d0) * aw);    // w^3 (s xi^2 + d0 q)
    const float R = f_rcp(den);
    const float hR = hgt * R;
    const float o = fmaf(hR, num, yk);
    const float M3 = fmaf(w, fmaf(d0 * wa, wa, (d1 * a) * a), h2 * aw);   // w^3 (d1 xi^2 + 2 s q + d0 (1-xi)^2)
    const float arg = (hR * hR) * (M3 * w);               // s^2 M / (s + t1 q)^2
    out = inb ? o : v;
    ld2 = f_lg2(inb ? arg : 1.0f);
}

// Inverse map (rational_quadratic.py:153-181).  out = spline^{-1}(v), ld2 = -log2 |d spline / d x| at out.
// LD = false: out only, ld2 is not written.
template <bool SAFE, int NY, bool DPOLY = false, bool LD = true>
B2F_HD void inverse(float v, const float (&g)[24], float b, float& out, float& ld2) {
    const float two_b = b + b;
    const bool inb = fabsf(v) < b;
    const float t = v + b;
    Sel s;
    select<true, SAFE, NY, DPOLY>(g, t, two_b, s);
    const float w = s.xu - s.xl, hgt = s.yu - s.yl;
    const float xk = s.xl - b;
    const float t0 = fminf(fmaxf(t - s.yl, 0.0f), hgt);   // v - y_k
    const f2 dd = knot_deltas<DPOLY>(s);
    const float d0 = dd.x, d1 = dd.y;
    const float h2 = hgt + hgt, hw = hgt * w;
    const float T = fmaf(w, d0 + d1, -h2);                // w * t1
    // quadratic of :170-178 multiplied by w:  A = hgt^2 - B,  B = hgt d0 w - t0 T,  C = -hgt t0
    const float B2 = fmaf(-t0, T, hw * d0);
    const float A2 = fmaf(hgt, hgt, -B2);
    const float disc = fmaf(B2, B2, (4.0f * (A2 * hgt)) * t0);
    const float sq = f_sqrt(fmaxf(disc, 0.0f));
    const float xi = fminf(fmaxf((h2 * t0) * f_rcp(B2 + sq), 0.0f), 1.0f);
    const float o = fmaf(xi, w, xk);                      // one explicit FMA: the same rounding with and without LD
    out = inb ? o : v;
    if (!LD) return;
    const float a = xi * w;
    const float wa = w - a, aw = a * wa;
    const float den = fmaf(T, aw, hw * w);
    const float M3 = fmaf(w, fmaf(d0 * wa, wa, (d1 * a) * a), h2 * aw);
    const float fw = (hgt * hgt) * (M3 * w);              // forward derivative = fw / den^2
    ld2 = f_lg2(inb ? den * den : 1.0f) - f_lg2(inb ? fw : 1.0f);
}


B2F_HD float f_rcpn(float x) {            // reciprocal + one Newton step (~1 ulp)
    const float y = f_rcp(x);
    return fmaf(y, fmaf(-x, y, 1.0f), y);
}

// ---- sequential direction of a masked autoregressive spline layer (b2f_flow_rows.cuh, rows_sequential_rq) --------------------
// One element per step with the SAME parameters used twice: the map itself, and -- for every dimension but the last -- the
// log-determinant the reference reports, which is the one of its last full pass, where the dimension is fed its already
// transformed value (layers_base.py:218-223, SURVEY Appendix B.3).  The softmax bin sizes are computed once (sizes), the bin
// search and the evaluation run per evaluation point (search / eval).  Same arithmetic as select / forward / inverse above
// (knot exponentials: see FASTEXP).
// FASTEXP: SFU exponentials (2 ulp: knots then differ from the one-pass direction's by ~1e-5 at boundary 50, which shows in the
// forward-then-inverse round trip); otherwise the ~1 ulp polynomial of b2f_math.cuh (the default: round trips stay at the
// reference's own level)
template <bool SAFE, bool FASTEXP>
B2F_HD void sizes(const float (&g)[24], float two_b, f2 (&sz)[8]) {
    f2 e[8];
    float m = 0.0f, my = 0.0f;
    if (SAFE) {
        m = g[0]; my = g[0] + g[8];
#pragma unroll
        for (int j = 1; j < 8; ++j) { m = fmaxf(m, g[j]); my = fmaxf(my, g[j] + g[8 + j]); }
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        const float ax = SAFE ? g[j] - m : g[j], ay = SAFE ? (g[j] + g[8 + j]) - my : g[j] + g[8 + j];
        if (FASTEXP) { e[j].x = f_ex2(ax); e[j].y = f_ex2(ay); }
        else e[j] = exp_det2(mk2(ax * kLn2, ay * kLn2));
    }
    const f2 sum = pk_add(pk_add(pk_add(e[0], e[1]), pk_add(e[2], e[3])), pk_add(pk_add(e[4], e[5]), pk_add(e[6], e[7])));
    const float r = (kSizeScale * two_b) * f_rcpn(sum.x * sum.y);     // Newton-refined: errors feed the next dimensions
    const f2 rr = mk2(r * sum.y, r * sum.x);
    const float minb = kRqMinBin * two_b;
#pragma unroll
    for (int j = 0; j < 8; ++j) sz[j] = pk_fma(e[j], rr, mk2(minb, minb));
}

template <bool INV>
B2F_HD void search(const f2 (&sz)[8], const float (&g)[24], float t, float two_b, Sel& s) {
    f2 lo = mk2(0.0f, 0.0f), up = sz[0];
    s.dl0 = kEdgeLogit; s.dl1 = kEdgeLogit + g[16];
    float c = 0.0f, m7 = 0.0f;
#pragma unroll
    for (int j = 1; j < 8; ++j) {
        c += INV ? sz[j - 1].y : sz[j - 1].x;
        m7 = select_step(c, t, lo, up, s.dl0, s.dl1, sz[j - 1], sz[j], g[16 + j - 1], g[16 + j]);
    }
    if (m7 != 0.0f) up = mk2(two_b, two_b);
    s.xl = lo.x; s.yl = lo.y; s.xu = up.x; s.yu = up.y;
}

// value and log2 |d out / d v| of the map at t = v + b inside the selected bin (no bounds handling)
template <bool INV>
B2F_HD void eval(float t, const Sel& s, float b, float& o, float& ld2) {
    const float w = s.xu - s.xl, hgt = s.yu - s.yl;
    const float d0 = delta(s.dl0), d1 = delta(s.dl1);
    const float h2 = hgt + hgt, hw = hgt * w;
    const float T = fmaf(w, d0 + d1, -h2);
    if (!INV) {
        const float a = fminf(fmaxf(t - s.xl, 0.0f), w);
        const float wa = w - a, aw = a * wa;
        const float den = fmaf(T, aw, hw * w);
        const float num = fmaf(hgt * a, a, (w * d0) * aw);
        const float hR = hgt * f_rcpn(den);
        o = fmaf(hR, num, s.yl - b);
        const float M3 = fmaf(w, fmaf(d0 * wa, wa, (d1 * a) * a), h2 * aw);
        ld2 = f_lg2((hR * hR) * (M3 * w));
    } else {
        const float t0 = fminf(fmaxf(t - s.yl, 0.0f), hgt);
        const float B2 = fmaf(-t0, T, hw * d0);
        const float A2 = fmaf(hgt, hgt, -B2);
        const float disc = fmaf(B2, B2, (4.0f * (A2 * hgt)) * t0);
        const float sq = sqrtf(fmaxf(disc, 0.0f));
        const float xi = fminf(fmaxf((h2 * t0) * f_rcpn(B2 + sq), 0.0f), 1.0f);
        const float a = xi * w;
        o = (s.xl - b) + a;
        const float wa = w - a, aw = a * wa;
        const float den = fmaf(T, aw, hw * w);
        const float M3 = fmaf(w, fmaf(d0 * wa, wa, (d1 * a) * a), h2 * aw);
        ld2 = f_lg2(den * den) - f_lg2((hgt * hgt) * (M3 * w));
    }
}

// out = map(v); ld2 = log2-determinant of the map evaluated AT out (QUIRK, see above) or at v (the exact one)
template <bool INV, bool SAFE, bool QUIRK, bool FASTEXP>
B2F_HD void sequential_step(float v, const float (&g)[24], float b, float& out, float& ld2) {
    const float two_b = b + b;
    const bool inb = fabsf(v) < b;
    f2 sz[8];
    sizes<SAFE, FASTEXP>(g, two_b, sz);
    Sel s;
    search<INV>(sz, g, v + b, two_b, s);
    float o, l;
    eval<INV>(v + b, s, b, o, l);
    out = inb ? o : v;
    if (QUIRK) {
        const bool inb2 = inb && fabsf(out) < b;
        search<INV>(sz, g, out + b, two_b, s);
        float o2, l2;
        eval<INV>(out + b, s, b, o2, l2);
        ld2 = inb2 ? l2 : 0.0f;
    } else {
        ld2 = inb ? l : 0.0f;
    }
}


// ---- backward of the forward-direction spline on the RAW 23 parameters (p[0..8) widths logits, p[8..16) heights
// offsets, p[16..23) interior derivative logits; p[23] unused) for the wide-conditioner kernel (b2f_wide.cu), whose
// backward is the epilogue of a GEMM and must be short.  Same partial derivatives as rq_backward_fwd (b2f_math.cuh,
// SURVEY Appendix D), restructured: the two softmaxes are evaluated ONCE (SFU ex2, shared by the knots and by the softmax
// backward -- rq_backward_fwd evaluates 32 polynomial exponentials), reciprocals instead of divisions, the sigmoid of the
// two selected derivative logits only.  ~450 issue slots instead of ~1700.  Tolerance-checked against rq_backward_fwd
// (tests/test_c_oracle_and_hostmath.py) like everything downstream of a TF32 GEMM.

B2F_HD void backward_fwd(float v, const float (&p)[24], float b, float GZ_in, float GL_in, float& dv, float (&dp)[24]) {
    // Out of bounds (identity tail): dL/dv = GZ and zero parameter gradients.  The arithmetic below runs on v clamped into
    // the spline's range with the upstream gradients zeroed, so it stays finite and every product with them is an exact 0.
    const bool inb = v > -b && v < b;
    const float lo = -b, span = b + b;
    const float vc = fminf(fmaxf(v, lo), b);
    const float GZ = inb ? GZ_in : 0.0f, GL = inb ? GL_in : 0.0f;
    // softmaxes (rational_quadratic.py:75-76, 46-47); cx = c1 * softmax (c1 = 1 - 8e-3), the form both the bin sizes and the
    // softmax backward use
    float cx[8], cy[8];
    float mx = p[0], my = fmaf(p[8], 1e-3f, p[0]);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        cx[j] = p[j];
        cy[j] = fmaf(p[8 + j], 1e-3f, p[j]);
        mx = fmaxf(mx, cx[j]);
        my = fmaxf(my, cy[j]);
    }
    float sx = 0.0f, sy = 0.0f;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        cx[j] = f_ex2((cx[j] - mx) * kLog2e);
        cy[j] = f_ex2((cy[j] - my) * kLog2e);
        sx += cx[j];
        sy += cy[j];
    }
    const float isx = kSizeScale * f_rcpn(sx), isy = kSizeScale * f_rcpn(sy);
    // Search with the predicates as numbers.  m_j = [knot_{j+1} < v] (searchsorted right=False), M_j = [knot_j < v] = m_{j-1}
    // (M_0 = 1), d_j = M_j - m_j = [bin j is the one].  Monotone predicates make the predicated prefix sums EXACTLY the
    // cumulative sums of the selected knots, in the reference's summation order; knot = span * cumsum + lo.
    float m[8], d[8];
    float Cx = 0.0f, Cx1 = 0.0f, Cy = 0.0f, Cy1 = 0.0f, ud0 = 0.0f, ud1 = 0.0f, c = 0.0f, Mj = 1.0f;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        cx[j] *= isx;
        cy[j] *= isy;
        const float wx = cx[j] + kRqMinBin, wy = cy[j] + kRqMinBin;      // bin sizes in units of the range
        c += wx;
        m[j] = (j < 7 && fmaf(span, c, lo) < vc) ? 1.0f : 0.0f;          // knot 8 = +b is never below v
        d[j] = Mj - m[j];
        Cx = fmaf(m[j], wx, Cx);  Cx1 = fmaf(Mj, wx, Cx1);
        Cy = fmaf(m[j], wy, Cy);  Cy1 = fmaf(Mj, wy, Cy1);
        const float aj = j == 0 ? kRqEdgeU : p[16 + (j == 0 ? 0 : j - 1)];       // derivative logit of knot j
        const float aj1 = j == 7 ? kRqEdgeU : p[16 + (j == 7 ? 0 : j)];          // ... of knot j + 1
        ud0 = fmaf(d[j], aj, ud0);
        ud1 = fmaf(d[j], aj1, ud1);
        Mj = m[j];
    }
    const float xk = fmaf(span, Cx, lo), yk = fmaf(span, Cy, lo);
    const float xk1 = d[7] != 0.0f ? b : fmaf(span, Cx1, lo), yk1 = d[7] != 0.0f ? b : fmaf(span, Cy1, lo);    // knot 8 is pinned
    // evaluation inside the bin (rational_quadratic.py:88-109)
    const float w = xk1 - xk, hgt = yk1 - yk;
    const float iw = f_rcpn(w);
    const float sk = hgt * iw;
    const float xr = (vc - xk) * iw;
    const float a0 = fmaf(ud0, 1e-3f, kRqEdgeU), a1 = fmaf(ud1, 1e-3f, kRqEdgeU);
    const float e0 = f_ex2(a0 * kLog2e), e1 = f_ex2(a1 * kLog2e);
    const float d0 = fmaf(f_lg2(1.0f + e0), kLn2, kRqMinDelta), d1 = fmaf(f_lg2(1.0f + e1), kLn2, kRqMinDelta);
    const float t1 = d1 + d0 - 2.0f * sk;
    const float xi = fminf(fmaxf(xr, 0.0f), 1.0f);
    const bool clipped = (xr < 0.0f) || (xr > 1.0f);
    const float omx = 1.0f - xi;
    const float q = xi * omx;
    const float Dn = fmaf(t1, q, sk);
    const float M = fmaf(d1 * xi, xi, fmaf(2.0f * sk, q, d0 * omx * omx));
    const float iDn = f_rcpn(Dn), iM = f_rcpn(M), isk = f_rcpn(sk);
    const float A = fmaf(sk * xi, xi, d0 * q);
    const float omq = 1.0f - 2.0f * q, om2x = 1.0f - 2.0f * xi;
    const float hD2 = hgt * iDn * iDn;
    // partials (Appendix D)
    const float out_xi = hD2 * sk * M;
    const float out_s = hD2 * fmaf(xi * xi, Dn, -A * omq);
    const float out_d0 = hD2 * q * (Dn - A);
    const float out_d1 = -hD2 * A * q;
    const float ld_xi = 2.0f * (fmaf(d1, xi, fmaf(sk, om2x, -d0 * omx)) * iM - t1 * om2x * iDn);
    const float ld_s = 2.0f * (isk + q * iM - omq * iDn);
    const float ld_d0 = fmaf(omx * omx, iM, -2.0f * q * iDn);
    const float ld_d1 = fmaf(xi * xi, iM, -2.0f * q * iDn);
    float Gxi = fmaf(GZ, out_xi, GL * ld_xi);
    if (clipped) Gxi = 0.0f;
    const float Gs = fmaf(GZ, out_s, GL * ld_s);
    const float dvi = Gxi * iw;
    const float Gw = -(fmaf(Gxi, xi, Gs * sk)) * iw;
    const float Ghgt = fmaf(GZ * A, iDn, Gs * iw);
    const float Gd0 = fmaf(GZ, out_d0, GL * ld_d0), Gd1 = fmaf(GZ, out_d1, GL * ld_d1);
    // softmax backward: knot gradients g_j = span (m_j G_below + d_j G_at); J(p, g)_j = c1 p_j (g_j - sum_i p_i g_i)
    const float sGxk = -span * dvi, sGw = span * Gw, sGyk = span * GZ, sGh = span * Ghgt;
    float gx[8], gy[8];
    float dotx = 0.0f, doty = 0.0f;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        gx[j] = fmaf(m[j], sGxk, d[j] * sGw);
        gy[j] = fmaf(m[j], sGyk, d[j] * sGh);
        dotx = fmaf(cx[j], gx[j], dotx);
        doty = fmaf(cy[j], gy[j], doty);
    }
    dotx *= 1.0f / kSizeScale;                    // cx carries c1: sum_i p_i g_i = dot / c1
    doty *= 1.0f / kSizeScale;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        const float jx = cx[j] * (gx[j] - dotx);
        const float jy = cy[j] * (gy[j] - doty);
        dp[j] = jx + jy;
        dp[8 + j] = jy * 1e-3f;
    }
    // derivative logits: softplus' = sigmoid = e / (1 + e); only knots k (lower) and k + 1 (upper) receive anything
    const float g0 = Gd0 * e0 * f_rcpn(1.0f + e0) * 1e-3f, g1 = Gd1 * e1 * f_rcpn(1.0f + e1) * 1e-3f;
#pragma unroll
    for (int jj = 1; jj < 8; ++jj) dp[16 + jj - 1] = fmaf(d[jj], g0, d[jj - 1] * g1);
    dp[23] = 0.0f;
    dv = inb ? dvi : GZ_in;
}

}  // namespace rqf
}  // namespace b2f
