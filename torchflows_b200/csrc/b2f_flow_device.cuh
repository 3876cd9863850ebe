// Device-side building blocks shared by the forward flow kernel (b2f_flow.cu) and the backward flow kernel
// (b2f_flow_bwd.cu): op descriptors, the shared-memory tile view, the conditioner's two layers and the
// transformer dispatch.  See b2f_flow.cu for the layout and thread-mapping rationale.
#pragma once
#include "b2f_common.cuh"
#include "b2f_math.cuh"
#include "b2f_lrs.cuh"

namespace b2f {

struct DevOp {
    int kind, tkind, H, flags;
    float boundary;
    int pad_;
    const float *p0, *p1, *p2, *p3;
    const int* p4;
};

template <int TK> struct TInfo;
template <> struct TInfo<B2F_T_SHIFT_ADD> { static constexpr int P = 1, PP = 1; };
template <> struct TInfo<B2F_T_SHIFT_SUB> { static constexpr int P = 1, PP = 1; };
template <> struct TInfo<B2F_T_AFFINE_FWD> { static constexpr int P = 2, PP = 2; };
template <> struct TInfo<B2F_T_AFFINE_INV> { static constexpr int P = 2, PP = 2; };
template <> struct TInfo<B2F_T_RQ_FWD> { static constexpr int P = 23, PP = 24; };
template <> struct TInfo<B2F_T_RQ_INV> { static constexpr int P = 23, PP = 24; };
template <> struct TInfo<B2F_T_LRS_FWD> { static constexpr int P = 32, PP = 32; };     // LinearRational, n_bins 8: 4 * 8
template <> struct TInfo<B2F_T_LRS_INV> { static constexpr int P = 32, PP = 32; };

// transformer kinds whose sequential direction reports the reference's last-iteration log-det (SURVEY Appendix B.3)
template <int TK> constexpr bool kSplineTk = TK == B2F_T_RQ_FWD || TK == B2F_T_RQ_INV || TK == B2F_T_LRS_FWD || TK == B2F_T_LRS_INV;

// transformer parameters of one element from the hidden activations of this thread's sample:
// acc[p] = b2[e*P+p] + sum_j W2tile[e][j][p] * hid[j]          (transforms.py:297-300, last Linear)
template <int P, int PP, bool GLOBAL = true>
__device__ __forceinline__ void element_params(float (&acc)[PP], const float* __restrict__ w2e,
                                               const float* __restrict__ b2e, const float* hid_m, int H) {
    // GLOBAL: the weights are read through the read-only path (ld.global.nc); otherwise they sit in shared memory
    auto ld1 = [](const float* q) { if constexpr (GLOBAL) return __ldg(q); else return *q; };
    auto ld2 = [](const float2* q) { if constexpr (GLOBAL) return __ldg(q); else return *q; };
    auto ld4 = [](const float4* q) { if constexpr (GLOBAL) return __ldg(q); else return *q; };
#pragma unroll
    for (int p = 0; p < PP; ++p) acc[p] = (p < P) ? ld1(b2e + p) : 0.0f;
    if constexpr (PP % 4 == 0) {
        const float4* w = reinterpret_cast<const float4*>(w2e);
        for (int j = 0; j < H; ++j) {
            const float hj = hid_m[j];
#pragma unroll
            for (int c = 0; c < PP / 4; ++c) {
                const float4 wv = ld4(w + j * (PP / 4) + c);
                acc[4 * c + 0] = fmaf(wv.x, hj, acc[4 * c + 0]);
                acc[4 * c + 1] = fmaf(wv.y, hj, acc[4 * c + 1]);
                acc[4 * c + 2] = fmaf(wv.z, hj, acc[4 * c + 2]);
                acc[4 * c + 3] = fmaf(wv.w, hj, acc[4 * c + 3]);
            }
        }
    } else if constexpr (PP == 2) {
        const float2* w = reinterpret_cast<const float2*>(w2e);
        for (int j = 0; j < H; ++j) {
            const float hj = hid_m[j];
            const float2 wv = ld2(w + j);
            acc[0] = fmaf(wv.x, hj, acc[0]);
            acc[1] = fmaf(wv.y, hj, acc[1]);
        }
    } else {
        for (int j = 0; j < H; ++j) acc[0] = fmaf(ld1(w2e + j), hid_m[j], acc[0]);
    }
}

template <int TK, int MODE, int PP>
__device__ __forceinline__ void transform_element(float v, const float (&acc)[PP], float boundary, float& out,
                                                  float& ld) {
    if constexpr (TK == B2F_T_SHIFT_ADD) { out = v + acc[0]; ld = 0.0f; }
    else if constexpr (TK == B2F_T_SHIFT_SUB) { out = v - acc[0]; ld = 0.0f; }
    else if constexpr (TK == B2F_T_AFFINE_FWD) affine_fwd<MODE>(v, acc[0], acc[1], out, ld);
    else if constexpr (TK == B2F_T_AFFINE_INV) affine_inv<MODE>(v, acc[0], acc[1], out, ld);
    else if constexpr (TK == B2F_T_LRS_FWD || TK == B2F_T_LRS_INV) {
        // linear rational spline (csrc/b2f_lrs.cuh): libm arithmetic in every mode
        auto h = [&](int i) { return acc[i]; };
        lrs_apply<8, TK == B2F_T_LRS_INV>(v, h, 8, boundary, out, ld);
    } else {
        int k;
        auto h = [&](int i) { return acc[i]; };
        rq_apply<8, TK == B2F_T_RQ_INV, MODE>(v, h, 8, boundary, out, ld, k);
    }
}

struct Tile {
    float* xt;   // [TM][XS]
    float* hid;  // [TM][HS]   hidden activations (or pre-activations in the sequential op)
    float* act;  // [TM][HS]   sequential op only
    float* ldp;  // [WPG][TM]  log-det partials per element slot
    int D, TM, logTM, XS, HS, WPG, G;
    int flip;    // logical column j lives at physical column (flip ? D-1-j : j)
    __device__ __forceinline__ int col(int j) const { return flip ? D - 1 - j : j; }
};

// hidden layer: hid[m][j] = act(b1[j] + sum_k W1[j][k] * x[m][src k])     (transforms.py:295-296 / :259-262)
// row_bias: per-row hidden bias of this tile's rows ([TM][H], B2F_FLAG_ROW_BIAS: context-conditioned layer), else nullptr;
// rows: valid rows of the tile (rows beyond it get a zero bias, their results are never stored).
template <bool TANH>
__device__ __forceinline__ void hidden_layer(const Tile& t, const DevOp& op, int n_src, const float* row_bias = nullptr,
                                             int rows = 0) {
    const int H = op.H;
    for (int idx = threadIdx.x; idx < (H << t.logTM); idx += blockDim.x) {
        const int m = idx & (t.TM - 1), j = idx >> t.logTM;   // j is warp-uniform: W1 reads are broadcasts
        const float* w = op.p0 + (size_t)j * n_src;
        const float* xr = t.xt + m * t.XS;
        float a0 = row_bias ? (m < rows ? __ldg(row_bias + (size_t)m * H + j) : 0.0f) : __ldg(op.p1 + j), a1 = 0.0f;
        int k = 0;
        if (!t.flip) {
            for (; k + 1 < n_src; k += 2) {
                a0 = fmaf(__ldg(w + k), xr[k], a0);
                a1 = fmaf(__ldg(w + k + 1), xr[k + 1], a1);
            }
            if (k < n_src) a0 = fmaf(__ldg(w + k), xr[k], a0);
        } else {
            const float* xe = xr + t.D - 1;
            for (; k + 1 < n_src; k += 2) {
                a0 = fmaf(__ldg(w + k), xe[-k], a0);
                a1 = fmaf(__ldg(w + k + 1), xe[-k - 1], a1);
            }
            if (k < n_src) a0 = fmaf(__ldg(w + k), xe[-k], a0);
        }
        const float a = a0 + a1;
        t.hid[m * t.HS + j] = TANH ? tanhf(a) : a;
    }
}


// conditioner output layer + transformer for every target element (one pass)
template <int TK, int MODE>
__device__ __forceinline__ void transform_pass(const Tile& t, const DevOp& op, int t0, int n_tgt) {
    constexpr int P = TInfo<TK>::P, PP = TInfo<TK>::PP;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int g = warp % t.G, slot = warp / t.G;
    const int m = g * 32 + lane;
    const float* hid_m = t.hid + m * t.HS;
    float* xr = t.xt + m * t.XS;
    float ldpart = 0.0f;
    if (slot < t.WPG) {
        for (int e = slot; e < n_tgt; e += t.WPG) {
            float acc[PP];
            element_params<P, PP>(acc, op.p2 + (size_t)e * op.H * PP, op.p3 + (size_t)e * P, hid_m, op.H);
            const int c = t.col(t0 + e);
            float out, ld;
            transform_element<TK, MODE, PP>(xr[c], acc, op.boundary, out, ld);
            xr[c] = out;
            ldpart += ld;
        }
        t.ldp[slot * t.TM + m] = ldpart;
    }
}

// D-step sequential direction of a masked autoregressive layer (layers_base.py:213-223) at the cost of ONE
// conditioner pass: hidden pre-activations are updated incrementally (rank-1 update per finished dimension)
// and only the P parameters of dimension i are evaluated at step i.  A thread owns a sample for all D steps.
template <int TK, int MODE>
__device__ __forceinline__ void sequential_pass(const Tile& t, const DevOp& op) {
    constexpr int P = TInfo<TK>::P, PP = TInfo<TK>::PP;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int g = warp % t.G, slot = warp / t.G;
    if (slot != 0) return;
    const int m = g * 32 + lane, H = op.H, D = t.D;
    float* pre = t.hid + m * t.HS;
    float* act = t.act + m * t.HS;
    float* xr = t.xt + m * t.XS;
    for (int j = 0; j < H; ++j) { pre[j] = __ldg(op.p1 + j); act[j] = 0.0f; }
    const bool quirk = kSplineTk<TK> && !(op.flags & B2F_FLAG_SEQ_LOGDET_EXACT);
    float ldsum = 0.0f;
    for (int i = 0; i < D; ++i) {
        // hidden units whose inputs x_0..x_{i-1} are now all final
        for (int j = 0; j < H; ++j)
            if (__ldg(op.p4 + j) == i) act[j] = tanhf(pre[j]);
        float acc[PP];
        element_params<P, PP>(acc, op.p2 + (size_t)i * H * PP, op.p3 + (size_t)i * P, act, H);
        const int c = t.col(i);
        float out, ld;
        transform_element<TK, MODE, PP>(xr[c], acc, op.boundary, out, ld);
        if (quirk && i < D - 1) {
            // The reference returns the log-det of its LAST full pass, in which dimension i < D-1 is fed the
            // already inverted value (layers_base.py:218-223, SURVEY Appendix B.3): reproduce that term.
            float out2;
            transform_element<TK, MODE, PP>(out, acc, op.boundary, out2, ld);
        }
        xr[c] = out;
        ldsum += ld;
        const float* w1c = op.p0 + i;    // column i of the (masked) first layer
        for (int j = 0; j < H; ++j) pre[j] = fmaf(__ldg(w1c + (size_t)j * D), out, pre[j]);
    }
    t.ldp[m] = ldsum;
}

// ElementwiseAffine / ActNorm: global parameters value:(D,2) broadcast over the batch (layers_base.py:300-303).
// stage: ea[j] = alpha_j, ea[D+j] = beta_j, ea[2D+j] = log alpha_j;  apply: z = a*x + b  or  z = (x - b)/a.
__device__ __forceinline__ void elementwise_stage(float* ea, const DevOp& op, int D) {
    for (int j = threadIdx.x; j < D; j += blockDim.x) {
        float a, la;
        affine_scale<0>(__ldg(op.p0 + 2 * j), a, la);
        ea[j] = a; ea[D + j] = __ldg(op.p0 + 2 * j + 1); ea[2 * D + j] = la;
    }
}
__device__ __forceinline__ void elementwise_apply(const Tile& t, const float* ea, bool fwd) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, NW = blockDim.x >> 5, D = t.D;
    for (int m = warp; m < t.TM; m += NW) {
        float* xr = t.xt + m * t.XS;
        for (int j = lane; j < D; j += 32) {
            const int c = t.col(j);
            xr[c] = fwd ? fmaf(ea[j], xr[c], ea[D + j]) : (xr[c] - ea[D + j]) / ea[j];
        }
    }
}

// A run of consecutive elementwise layers is ONE affine map per column, z = A_j*x + B_j (composition of
// a*x+b and (x-b)/a steps); the batch-independent log-det of the run is sum_j L_j.  `get(i)` returns the
// (kind, tkind, value pointer) of op i.  Stages ea[j] = A_j, ea[D+j] = B_j, ea[2D+j] = L_j and returns how many
// ops the run covers (>= 1).
struct EwOp { int kind, tkind; const float* value; };
template <class Get>
__device__ __forceinline__ int elementwise_stage_run(float* ea, const Get& get, int oi, int n_ops, int D, int tid, int nthreads) {
    int n_run = 1;
    while (oi + n_run < n_ops && get(oi + n_run).kind == B2F_OP_ELEMENTWISE) ++n_run;
    for (int j = tid; j < D; j += nthreads) {
        float Aj = 1.0f, Bj = 0.0f, Lj = 0.0f;
        for (int r = 0; r < n_run; ++r) {
            const EwOp o = get(oi + r);
            float a, la;
            affine_scale<0>(__ldg(o.value + 2 * j), a, la);
            const float b = __ldg(o.value + 2 * j + 1);
            if (o.tkind == B2F_T_AFFINE_FWD) { Aj *= a; Bj = fmaf(a, Bj, b); Lj += la; }
            else { const float ia = 1.0f / a; Aj *= ia; Bj = (Bj - b) * ia; Lj -= la; }
        }
        ea[j] = Aj; ea[D + j] = Bj; ea[2 * D + j] = Lj;
    }
    return n_run;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

}  // namespace b2f
