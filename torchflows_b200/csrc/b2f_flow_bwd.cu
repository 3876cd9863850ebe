// Backward of the fused flow program (kernel K6): one launch per call, no materialised h.
//
// Replaces torch autograd through the ~470-op graph the reference builds for one log_prob call
// (/root/reference/torchflows/flows.py:199-224 -> bijections/base.py:203-224 -> layers_base.py:145-153,
//  202-211, 300-318 -> transforms.py:293-307 -> transformers/...).  The math of the transformer backward is
// SURVEY.md Appendix D (csrc/b2f_math.cuh: rq_backward_fwd, affine_*_backward; csrc/b2f_lrs.cuh: lrs_backward).
//
// Per CTA (tile of TM samples, both the activation tile xt and the gradient tile gt live in shared memory):
//   phase A  recompute the forward pass layer by layer; the tile as it enters each conditioner layer is written
//            to the caller's workspace (B*D floats per such layer) because spline layers cannot be un-done
//            exactly; elementwise layers are un-done in place during phase B instead;
//   phase B  walk the layers in reverse.  For a conditioner layer: reload its input tile, recompute the hidden
//            activations and, per (sample, target element), the P transformer parameters in registers; run the
//            transformer backward -> dL/dx_target and dL/dh[P]; push dL/dh through the last Linear
//            (dL/dhid via shared-memory atomics, dL/dW2 and dL/db2 by a per-warp [P x 32]x[32 x H] product
//            staged in shared memory), then tanh', the first Linear (dL/dW1, dL/db1) and dL/dx_source.
// Parameter gradients are accumulated into global fp32 buffers with red.global.add (one atomic per weight
// per tile); the caller zero-fills them.  Deterministic within a tile, atomic order across tiles.
#include <stdlib.h>
#include <string.h>

#include <algorithm>

#include "b2f_flow_device.cuh"
#include "b2f_rqfast.cuh"

namespace b2f {

struct BwdOp {
    DevOp f;
    float *g0, *g1, *g2, *g3;
    long long ws_off;   // float offset of this op's saved input in the workspace (-1: none)
};

struct BwdArgs {
    BwdOp ops[B2F_MAX_OPS];
    int n_ops, D, TM, logTM, XS, HS, WPG, G, flags, wst_stride, dhs_pp;
    long long B;
    const float* x;
    const float* gy;
    const float* gld;
    const float* glp;
    const float* base_loc;
    const float* base_log_scale;
    float* gx;
    float* ws;
};

struct BTile {
    Tile t;
    float* gt;    // [TM][XS] gradient w.r.t. the current activations
    float* dhid;  // [TM][HS] gradient w.r.t. hidden activations, then pre-activations
    float* dhp;   // [WPG][TM][HS] per-slot partial sums of dhid (a warp owns its (slot, 32 samples) slice: no atomics)
    float* GL;    // [TM]     dL/dlog_det of each sample (constant through the layers)
    float* dhs;   // [NW][32][dhs_pp] per-warp staging of dL/dh for the weight-gradient product (dhs_pp >= every PP)
    float* wst;   // [NW][2][wst_stride] per-warp double buffer of one element's output-layer weights (spline layers)
    int rows, precise, wst_stride;
};

template <int TK, int MODE, int P, int PP>
__device__ __forceinline__ void transformer_backward_element(float v, const float (&acc)[PP], float boundary, float GZ,
                                                             float GL, float& dv, float (&dh)[PP]) {
#pragma unroll
    for (int p = 0; p < PP; ++p) dh[p] = 0.0f;
    if constexpr (TK == B2F_T_SHIFT_ADD) { dv = GZ; dh[0] = GZ; }
    else if constexpr (TK == B2F_T_SHIFT_SUB) { dv = GZ; dh[0] = -GZ; }
    else if constexpr (TK == B2F_T_AFFINE_FWD) affine_fwd_backward<MODE>(v, acc[0], GZ, GL, dv, dh[0], dh[1]);
    else if constexpr (TK == B2F_T_AFFINE_INV) affine_inv_backward<MODE>(v, acc[0], acc[1], GZ, GL, dv, dh[0], dh[1]);
    else if constexpr (TK == B2F_T_RQ_FWD) {
        if constexpr (MODE >= 1 && PP == 24) {
            // default mode: the restructured backward (one evaluation of the two softmaxes shared by the knots and by their
            // gradients, SFU exponentials, reciprocals): ~2.5x fewer instructions, tolerance-checked against rq_backward_fwd
            rqf::backward_fwd(v, acc, boundary, GZ, GL, dv, dh);
        } else {
            auto h = [&](int i) { return acc[i]; };
            auto g = [&](int i, float val) { dh[i] = val; };
            rq_backward_fwd<8, MODE>(v, h, 8, boundary, GZ, GL, dv, g);
        }
    } else if constexpr (TK == B2F_T_LRS_FWD || TK == B2F_T_LRS_INV) {
        auto h = [&](int i) { return acc[i]; };
        auto g = [&](int i, float val) { dh[i] = val; };
        lrs_backward<8, TK == B2F_T_LRS_INV>(v, h, 8, boundary, GZ, GL, dv, g);
    } else {
        auto h = [&](int i) { return acc[i]; };
        auto g = [&](int i, float val) { dh[i] = val; };
        rq_backward_inv<8, MODE>(v, h, 8, boundary, GZ, GL, dv, g);
    }
}

// conditioner-layer backward for every target element
template <int TK, int MODE>
__device__ __forceinline__ void transform_pass_backward(const BTile& b, const BwdOp& op, int t0, int n_tgt) {
    constexpr int P = TInfo<TK>::P, PP = TInfo<TK>::PP;
    const Tile& t = b.t;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int g = warp % t.G, slot = warp / t.G;
    const int m = g * 32 + lane, H = op.f.H;
    const float* hid_m = t.hid + m * t.HS;
    const float* hid_g = t.hid + (g * 32) * t.HS;
    float* dhs = b.dhs + warp * 32 * PP;
    const float GLm = b.GL[m];
    const bool want_w = op.g2 != nullptr;
    float* dhp_m = b.dhp + ((size_t)slot * t.TM + m) * t.HS;
    for (int j = 0; j < H; ++j) dhp_m[j] = 0.0f;
    for (int e = slot; e < n_tgt; e += t.WPG) {
        const float* w2e = op.f.p2 + (size_t)e * H * PP;
        float acc[PP], dh[PP];
        element_params<P, PP>(acc, w2e, op.f.p3 + (size_t)e * P, hid_m, H);
        const int c = t.col(t0 + e);
        float dv;
        transformer_backward_element<TK, MODE, P, PP>(t.xt[m * t.XS + c], acc, op.f.boundary, b.gt[m * t.XS + c], GLm,
                                                      dv, dh);
        b.gt[m * t.XS + c] = dv;
        // dL/dhid[m][j] += sum_p dh[p] * W2[e][j][p]
        for (int j = 0; j < H; ++j) {
            float s = 0.0f;
#pragma unroll
            for (int p = 0; p < P; ++p) s = fmaf(dh[p], __ldg(w2e + j * PP + p), s);
            dhp_m[j] += s;
        }
        if (want_w) {
            // dL/dW2[e][j][p] += sum_m dh[m][p] * hid[m][j];  dL/db2[e][p] += sum_m dh[m][p]   (m over this warp)
            __syncwarp();
#pragma unroll
            for (int p = 0; p < PP; ++p) dhs[lane * PP + p] = dh[p];
            __syncwarp();
            for (int idx = lane; idx < H * PP; idx += 32) {
                const int j = idx / PP, p = idx - j * PP;
                if (p < P) {
                    float s = 0.0f;
                    for (int mm = 0; mm < 32; ++mm) s = fmaf(dhs[mm * PP + p], hid_g[mm * t.HS + j], s);
                    atomicAdd(op.g2 + ((size_t)e * H + j) * PP + p, s);
                }
            }
            if (lane < P) {
                float s = 0.0f;
                for (int mm = 0; mm < 32; ++mm) s += dhs[mm * PP + lane];
                atomicAdd(op.g3 + (size_t)e * P + lane, s);
            }
        }
    }
}

// ---- the same layer with its two batch-sized contractions on the tensor cores (spline layers, default arithmetic) ------
// Per warp (32 samples) and target element e, with dh[row][p] the transformer's parameter gradient (P = 23, padded 24):
//   dL/dW2[e][j][p] = sum_row hid[row][j] * dh[row][p]   (+ a constant-1 hidden row H for dL/db2[e][p])
//   dL/dhid[row][j] = sum_p   dh[row][p]  * W2[e][j][p]
// are [H+1 x 32] x [32 x 24] and [32 x 24] x [24 x H] products: mma.sync.m16n8k8 TF32 with fp32 accumulation, as the
// 3xTF32 split  a*b ~= a_lo*b_hi + a_hi*b_lo + a_hi*b_hi  (a_hi = the operand's upper 19 bits, which is what the tensor
// core reads from an fp32 register anyway; a_lo = a - a_hi, exact) -- fp32-faithful to ~2^-21, so the gradients keep the
// accuracy of the FFMA path above (`precise` mode and H > 31 still take that path).  dh goes through the per-warp staging
// buffer dhs[32][24] to reach the fragment layouts; the hid fragments are loaded once per layer; the dL/dhid accumulators
// live in registers across all elements of the warp.
__device__ __forceinline__ uint32_t tf32_hi(float x) { return __float_as_uint(x); }       // hardware ignores the low 13 bits
__device__ __forceinline__ uint32_t tf32_lo(float x) {
    return __float_as_uint(x - __uint_as_float(__float_as_uint(x) & 0xffffe000u));
}
__device__ __forceinline__ void mma3_tf32(float (&d)[4], const uint32_t (&ah)[4], const uint32_t (&al)[4], uint32_t bh0,
                                          uint32_t bh1, uint32_t bl0, uint32_t bl1);
__device__ __forceinline__ void mma_tf32(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
    asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                 : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
                 : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

__device__ __forceinline__ void mma3_tf32(float (&d)[4], const uint32_t (&ah)[4], const uint32_t (&al)[4], uint32_t bh0,
                                          uint32_t bh1, uint32_t bl0, uint32_t bl1) {
    mma_tf32(d, al, bh0, bh1);
    mma_tf32(d, ah, bl0, bl1);
    mma_tf32(d, ah, bh0, bh1);
}

// MT = ceil((H+1)/16) row tiles of dL/dW2^T, NT2 = ceil(H/8) column tiles of dL/dhid
template <int TK, int MODE, int MT, int NT2>
__device__ __forceinline__ void transform_pass_backward_mma(const BTile& b, const BwdOp& op, int t0, int n_tgt) {
    constexpr int P = TInfo<TK>::P, PP = TInfo<TK>::PP;
    static_assert(PP == 24, "spline layers only");
    const Tile& t = b.t;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int g = warp % t.G, slot = warp / t.G;
    const int m = g * 32 + lane, H = op.f.H;
    const int gq = lane >> 2, tq = lane & 3;
    const float* hid_m = t.hid + m * t.HS;
    const float* hid_g = t.hid + (g * 32) * t.HS;
    float* dhs = b.dhs + warp * 32 * PP;
    const float GLm = b.GL[m];
    const bool want_w = op.g2 != nullptr;

    // A fragments of dL/dW2^T = hid^T (rows j, columns = the warp's 32 samples), row H = 1 (bias), rows > H = 0
    float a1[MT][4][4];
    {
        auto hv = [&](int row, int j) { return j < H ? hid_g[row * t.HS + j] : (j == H ? 1.0f : 0.0f); };
#pragma unroll
        for (int mt = 0; mt < MT; ++mt)
#pragma unroll
            for (int ks = 0; ks < 4; ++ks) {
                a1[mt][ks][0] = hv(8 * ks + tq, 16 * mt + gq);
                a1[mt][ks][1] = hv(8 * ks + tq, 16 * mt + gq + 8);
                a1[mt][ks][2] = hv(8 * ks + tq + 4, 16 * mt + gq);
                a1[mt][ks][3] = hv(8 * ks + tq + 4, 16 * mt + gq + 8);
            }
    }
    float acc2[2][NT2][4];        // dL/dhid of the warp's 32 samples, summed over this warp's elements
#pragma unroll
    for (int mt = 0; mt < 2; ++mt)
#pragma unroll
        for (int nt = 0; nt < NT2; ++nt)
#pragma unroll
            for (int i = 0; i < 4; ++i) acc2[mt][nt][i] = 0.0f;

    // W2[e] (H x 24 floats) + b2[e] of the NEXT element travel global -> shared (cp.async) behind the current element's
    // math: with 8 warps per SM every weight load from L2 would otherwise be an exposed round trip (the j-loop of the
    // output layer alone is H dependent ones)
    float* wbuf[2] = {b.wst + (size_t)(2 * warp) * b.wst_stride, b.wst + (size_t)(2 * warp + 1) * b.wst_stride};
    auto stage = [&](int e, float* dst) {
        const float4* src = reinterpret_cast<const float4*>(op.f.p2 + (size_t)e * H * PP);
        for (int q = lane; q < H * (PP / 4); q += 32) {
            const unsigned d = (unsigned)__cvta_generic_to_shared(dst + 4 * q);
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d), "l"(src + q) : "memory");
        }
        if (lane < P) {
            const unsigned d = (unsigned)__cvta_generic_to_shared(dst + H * PP + lane);
            asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(d), "l"(op.f.p3 + (size_t)e * P + lane) : "memory");
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    };
    int cur = 0;
    if (slot < n_tgt) stage(slot, wbuf[0]);
    for (int e = slot; e < n_tgt; e += t.WPG, cur ^= 1) {
        asm volatile("cp.async.wait_group 0;" ::: "memory");
        __syncwarp();                  // this element's weights have landed; everyone is done with the other buffer
        const float* w2e = wbuf[cur];
        if (e + t.WPG < n_tgt) stage(e + t.WPG, wbuf[cur ^ 1]);
        {
            float acc[PP], dh[PP];
            {
                // transformer parameters of the warp's 32 samples: [32 x (H+1)] (hid | 1) times [(H+1) x 24] (W2[e] ; b2[e],
                // contiguous in the staged block) on the tensor cores (3xTF32), then through the staging buffer to get
                // from the accumulator layout to one sample per thread
                float pacc[2][3][4];
#pragma unroll
                for (int mt = 0; mt < 2; ++mt)
#pragma unroll
                    for (int nt = 0; nt < 3; ++nt)
#pragma unroll
                        for (int i = 0; i < 4; ++i) pacc[mt][nt][i] = 0.0f;
                auto hv = [&](int row, int j) { return j < H ? hid_g[row * t.HS + j] : (j == H ? 1.0f : 0.0f); };
#pragma unroll
                for (int ks = 0; ks < NT2; ++ks) {               // NT2 = ceil((H+1)/8) as well
                    uint32_t ah[2][4], al[2][4];
#pragma unroll
                    for (int mt = 0; mt < 2; ++mt) {
                        const float v[4] = {hv(16 * mt + gq, 8 * ks + tq), hv(16 * mt + gq + 8, 8 * ks + tq),
                                            hv(16 * mt + gq, 8 * ks + tq + 4), hv(16 * mt + gq + 8, 8 * ks + tq + 4)};
#pragma unroll
                        for (int i = 0; i < 4; ++i) { ah[mt][i] = tf32_hi(v[i]); al[mt][i] = tf32_lo(v[i]); }
                    }
#pragma unroll
                    for (int nt = 0; nt < 3; ++nt) {
                        const int j0 = 8 * ks + tq, j1 = j0 + 4;
                        const float w0 = j0 <= H ? w2e[j0 * PP + 8 * nt + gq] : 0.0f;
                        const float w1 = j1 <= H ? w2e[j1 * PP + 8 * nt + gq] : 0.0f;
#pragma unroll
                        for (int mt = 0; mt < 2; ++mt)
                            mma3_tf32(pacc[mt][nt], ah[mt], al[mt], tf32_hi(w0), tf32_hi(w1), tf32_lo(w0), tf32_lo(w1));
                    }
                }
#pragma unroll
                for (int mt = 0; mt < 2; ++mt)
#pragma unroll
                    for (int nt = 0; nt < 3; ++nt) {
                        float* r0 = dhs + (16 * mt + gq) * PP + 8 * nt + 2 * tq;
                        *reinterpret_cast<float2*>(r0) = make_float2(pacc[mt][nt][0], pacc[mt][nt][1]);
                        *reinterpret_cast<float2*>(r0 + 8 * PP) = make_float2(pacc[mt][nt][2], pacc[mt][nt][3]);
                    }
                __syncwarp();
                const float4* prow = reinterpret_cast<const float4*>(dhs + lane * PP);
#pragma unroll
                for (int q = 0; q < PP / 4; ++q) {
                    const float4 v = prow[q];
                    acc[4 * q] = v.x; acc[4 * q + 1] = v.y; acc[4 * q + 2] = v.z; acc[4 * q + 3] = v.w;
                }
            }
            const int c = t.col(t0 + e);
            float dv;
            transformer_backward_element<TK, MODE, P, PP>(t.xt[m * t.XS + c], acc, op.f.boundary, b.gt[m * t.XS + c], GLm,
                                                          dv, dh);
            b.gt[m * t.XS + c] = dv;
            __syncwarp();
            float4* drow = reinterpret_cast<float4*>(dhs + lane * PP);
#pragma unroll
            for (int q = 0; q < PP / 4; ++q) drow[q] = make_float4(dh[4 * q], dh[4 * q + 1], dh[4 * q + 2], dh[4 * q + 3]);
            __syncwarp();
        }
        // dL/dhid += dh [32 x 24] * W2[e]^T [24 x H]
#pragma unroll
        for (int ks = 0; ks < 3; ++ks) {
            uint32_t a2h[2][4], a2l[2][4];
#pragma unroll
            for (int mt = 0; mt < 2; ++mt) {
                const float* r0 = dhs + (16 * mt + gq) * PP + 8 * ks + tq;
                const float v[4] = {r0[0], r0[8 * PP], r0[4], r0[8 * PP + 4]};
#pragma unroll
                for (int i = 0; i < 4; ++i) { a2h[mt][i] = tf32_hi(v[i]); a2l[mt][i] = tf32_lo(v[i]); }
            }
#pragma unroll
            for (int nt = 0; nt < NT2; ++nt) {
                const int j = 8 * nt + gq;
                const float* wj = w2e + j * PP + 8 * ks + tq;
                const float w0 = j < H ? wj[0] : 0.0f, w1 = j < H ? wj[4] : 0.0f;
#pragma unroll
                for (int mt = 0; mt < 2; ++mt)
                    mma3_tf32(acc2[mt][nt], a2h[mt], a2l[mt], tf32_hi(w0), tf32_hi(w1), tf32_lo(w0), tf32_lo(w1));
            }
        }
        if (want_w) {
            // dL/dW2[e]^T (+ bias row) = hid^T [H+1 x 32] * dh [32 x 24]
            float acc1[MT][3][4];
#pragma unroll
            for (int mt = 0; mt < MT; ++mt)
#pragma unroll
                for (int nt = 0; nt < 3; ++nt)
#pragma unroll
                    for (int i = 0; i < 4; ++i) acc1[mt][nt][i] = 0.0f;
#pragma unroll
            for (int ks = 0; ks < 4; ++ks)
#pragma unroll
                for (int nt = 0; nt < 3; ++nt) {
                    const float* r0 = dhs + (8 * ks + tq) * PP + 8 * nt + gq;
                    const float d0 = r0[0], d1 = r0[4 * PP];
#pragma unroll
                    for (int mt = 0; mt < MT; ++mt) {
                        uint32_t ah[4], al[4];
#pragma unroll
                        for (int i = 0; i < 4; ++i) { ah[i] = tf32_hi(a1[mt][ks][i]); al[i] = tf32_lo(a1[mt][ks][i]); }
                        mma3_tf32(acc1[mt][nt], ah, al, tf32_hi(d0), tf32_hi(d1), tf32_lo(d0), tf32_lo(d1));
                    }
                }
            float* g2e = op.g2 + (size_t)e * H * PP;
            float* g3e = op.g3 + (size_t)e * P;
#pragma unroll
            for (int mt = 0; mt < MT; ++mt)
#pragma unroll
                for (int nt = 0; nt < 3; ++nt)
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        // row j < H of the product is dL/dW2[e][j][:], row H is dL/db2[e][:]: one predicated reduction
                        const int j = 16 * mt + gq + ((i & 2) ? 8 : 0), p = 8 * nt + 2 * tq + (i & 1);
                        float* dst = (j < H) ? g2e + j * PP + p : g3e + p;
                        if (p < P && j <= H) atomicAdd(dst, acc1[mt][nt][i]);
                    }
        }
    }
    // this warp's partial of dL/dhid: (slot, sample, j) has exactly one owner lane, no atomics
    float* dhp = b.dhp + ((size_t)slot * t.TM + g * 32) * t.HS;
#pragma unroll
    for (int mt = 0; mt < 2; ++mt)
#pragma unroll
        for (int nt = 0; nt < NT2; ++nt)
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const int row = 16 * mt + gq + ((i & 2) ? 8 : 0), j = 8 * nt + 2 * tq + (i & 1);
                if (j < H) dhp[row * t.HS + j] = acc2[mt][nt][i];
            }
}

// Backward of the D-step sequential direction x_i = T(z_i; h_i(x_0..x_{i-1})) (layers_base.py:213-223).  A thread owns
// a sample.  With act_j = tanh(pre_j(x)) recomputed from the complete x, walk i = D-1..0:
//   dL/dx_i (total) = upstream + sum_j W1m[j][i] * dpre_j      (hidden units that read x_i are final: fin_j > i)
//   (dL/dz_i, dL/dh_i) = transformer backward at (z_i, h_i);   dact_j += sum_p dh_i[p] * W2m[i][j][p]
// and dact_j becomes dpre_j = dact_j (1 - act_j^2) once every output that reads unit j has been processed (i + 1 ==
// fin_j).  Weight gradients of the output layer use the same per-warp staged product as the one-pass layers.
template <int TK, int MODE>
__device__ __forceinline__ void sequential_pass_backward(const BTile& b, const BwdOp& op, const float* __restrict__ z_saved) {
    constexpr int P = TInfo<TK>::P, PP = TInfo<TK>::PP;
    const Tile& t = b.t;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int g = warp % t.G, slot = warp / t.G;
    if (slot != 0) return;
    const int m = g * 32 + lane, H = op.f.H, D = t.D;
    float* act = t.hid + m * t.HS;
    float* dact = b.dhid + m * t.HS;
    const float* hid_g = t.hid + (g * 32) * t.HS;
    float* xr = t.xt + m * t.XS;
    float* gr = b.gt + m * t.XS;
    float* dhs = b.dhs + warp * 32 * PP;
    const bool live = m < b.rows;
    const float GLm = b.GL[m];
    const bool want_w = op.g2 != nullptr;
    for (int j = 0; j < H; ++j) {
        const float* w = op.f.p0 + (size_t)j * D;
        float a = __ldg(op.f.p1 + j);
        for (int k = 0; k < D; ++k) a = fmaf(__ldg(w + k), xr[t.col(k)], a);
        act[j] = tanhf(a);
        dact[j] = 0.0f;
    }
    for (int i = D - 1; i >= 0; --i) {
        for (int j = 0; j < H; ++j)
            if (__ldg(op.f.p4 + j) == i + 1) dact[j] *= (1.0f - act[j] * act[j]);
        const int c = t.col(i);
        float gx = gr[c];
        for (int j = 0; j < H; ++j) gx = fmaf(__ldg(op.f.p0 + (size_t)j * D + i), dact[j], gx);
        const float* w2e = op.f.p2 + (size_t)i * H * PP;
        float acc[PP], dh[PP];
        element_params<P, PP>(acc, w2e, op.f.p3 + (size_t)i * P, act, H);
        const float zi = live ? __ldg(z_saved + (size_t)m * D + c) : 0.0f;
        float dv;
        transformer_backward_element<TK, MODE, P, PP>(zi, acc, op.f.boundary, gx, GLm, dv, dh);
        gr[c] = dv;
        for (int j = 0; j < H; ++j) {
            float sacc = 0.0f;
#pragma unroll
            for (int p = 0; p < P; ++p) sacc = fmaf(dh[p], __ldg(w2e + j * PP + p), sacc);
            dact[j] += sacc;
        }
        if (want_w) {
            __syncwarp();
#pragma unroll
            for (int p = 0; p < PP; ++p) dhs[lane * PP + p] = dh[p];
            __syncwarp();
            for (int idx = lane; idx < H * PP; idx += 32) {
                const int j = idx / PP, p = idx - j * PP;
                if (p < P) {
                    float sacc = 0.0f;
                    for (int mm = 0; mm < 32; ++mm) sacc = fmaf(dhs[mm * PP + p], hid_g[mm * t.HS + j], sacc);
                    atomicAdd(op.g2 + ((size_t)i * H + j) * PP + p, sacc);
                }
            }
            if (lane < P) {
                float sacc = 0.0f;
                for (int mm = 0; mm < 32; ++mm) sacc += dhs[mm * PP + lane];
                atomicAdd(op.g3 + (size_t)i * P + lane, sacc);
            }
        }
    }
}

template <int TK, int MODE>
__device__ __forceinline__ void transform_pass_backward_rq(const BTile& b, const BwdOp& op, int t0, int n_tgt) {
    const int H = op.f.H;
    if (b.precise || H > 31 || b.wst_stride == 0) transform_pass_backward<TK, MODE>(b, op, t0, n_tgt);
    else if (H <= 7) transform_pass_backward_mma<TK, MODE, 1, 1>(b, op, t0, n_tgt);
    else if (H <= 15) transform_pass_backward_mma<TK, MODE, 1, 2>(b, op, t0, n_tgt);
    else if (H <= 23) transform_pass_backward_mma<TK, MODE, 2, 3>(b, op, t0, n_tgt);
    else transform_pass_backward_mma<TK, MODE, 2, 4>(b, op, t0, n_tgt);
}

template <int MODE>
__device__ __forceinline__ void run_transform_backward(const BTile& b, const BwdOp& op, int t0, int n_tgt) {
    switch (op.f.tkind) {
        case B2F_T_SHIFT_ADD: transform_pass_backward<B2F_T_SHIFT_ADD, MODE>(b, op, t0, n_tgt); break;
        case B2F_T_SHIFT_SUB: transform_pass_backward<B2F_T_SHIFT_SUB, MODE>(b, op, t0, n_tgt); break;
        case B2F_T_AFFINE_FWD: transform_pass_backward<B2F_T_AFFINE_FWD, MODE>(b, op, t0, n_tgt); break;
        case B2F_T_AFFINE_INV: transform_pass_backward<B2F_T_AFFINE_INV, MODE>(b, op, t0, n_tgt); break;
        case B2F_T_RQ_FWD: transform_pass_backward_rq<B2F_T_RQ_FWD, MODE>(b, op, t0, n_tgt); break;
        case B2F_T_RQ_INV: transform_pass_backward_rq<B2F_T_RQ_INV, MODE>(b, op, t0, n_tgt); break;
        case B2F_T_LRS_FWD: transform_pass_backward<B2F_T_LRS_FWD, MODE>(b, op, t0, n_tgt); break;
        case B2F_T_LRS_INV: transform_pass_backward<B2F_T_LRS_INV, MODE>(b, op, t0, n_tgt); break;
        default: break;
    }
}

template <int MODE>
__device__ __forceinline__ void run_sequential_backward(const BTile& b, const BwdOp& op, const float* z_saved) {
    switch (op.f.tkind) {
        case B2F_T_SHIFT_ADD: sequential_pass_backward<B2F_T_SHIFT_ADD, MODE>(b, op, z_saved); break;
        case B2F_T_SHIFT_SUB: sequential_pass_backward<B2F_T_SHIFT_SUB, MODE>(b, op, z_saved); break;
        case B2F_T_AFFINE_FWD: sequential_pass_backward<B2F_T_AFFINE_FWD, MODE>(b, op, z_saved); break;
        case B2F_T_AFFINE_INV: sequential_pass_backward<B2F_T_AFFINE_INV, MODE>(b, op, z_saved); break;
        case B2F_T_RQ_INV: sequential_pass_backward<B2F_T_RQ_INV, MODE>(b, op, z_saved); break;
        case B2F_T_LRS_INV: sequential_pass_backward<B2F_T_LRS_INV, MODE>(b, op, z_saved); break;
        default: break;
    }
}

template <int MODE>
__device__ __forceinline__ void run_sequential_forward(const Tile& t, const DevOp& op) {
    switch (op.tkind) {
        case B2F_T_SHIFT_ADD: sequential_pass<B2F_T_SHIFT_ADD, MODE>(t, op); break;
        case B2F_T_SHIFT_SUB: sequential_pass<B2F_T_SHIFT_SUB, MODE>(t, op); break;
        case B2F_T_AFFINE_FWD: sequential_pass<B2F_T_AFFINE_FWD, MODE>(t, op); break;
        case B2F_T_AFFINE_INV: sequential_pass<B2F_T_AFFINE_INV, MODE>(t, op); break;
        case B2F_T_RQ_INV: sequential_pass<B2F_T_RQ_INV, MODE>(t, op); break;
        case B2F_T_LRS_INV: sequential_pass<B2F_T_LRS_INV, MODE>(t, op); break;
        default: break;
    }
}

template <int MODE>
__device__ __forceinline__ void run_transform_forward(const Tile& t, const DevOp& op, int t0, int n_tgt) {
    switch (op.tkind) {
        case B2F_T_SHIFT_ADD: transform_pass<B2F_T_SHIFT_ADD, MODE>(t, op, t0, n_tgt); break;
        case B2F_T_SHIFT_SUB: transform_pass<B2F_T_SHIFT_SUB, MODE>(t, op, t0, n_tgt); break;
        case B2F_T_AFFINE_FWD: transform_pass<B2F_T_AFFINE_FWD, MODE>(t, op, t0, n_tgt); break;
        case B2F_T_AFFINE_INV: transform_pass<B2F_T_AFFINE_INV, MODE>(t, op, t0, n_tgt); break;
        case B2F_T_RQ_FWD: transform_pass<B2F_T_RQ_FWD, MODE>(t, op, t0, n_tgt); break;
        case B2F_T_RQ_INV: transform_pass<B2F_T_RQ_INV, MODE>(t, op, t0, n_tgt); break;
        case B2F_T_LRS_FWD: transform_pass<B2F_T_LRS_FWD, MODE>(t, op, t0, n_tgt); break;
        case B2F_T_LRS_INV: transform_pass<B2F_T_LRS_INV, MODE>(t, op, t0, n_tgt); break;
        default: break;
    }
}

template <int MODE>
__global__ void __launch_bounds__(384) flow_backward_kernel(const __grid_constant__ BwdArgs A) {
    extern __shared__ __align__(16) float smem[];
#ifdef B2F_BWD_CLOCK_HOOK
    // Phase timing from inside the kernel (build with -DB2F_BWD_CLOCK_HOOK, run with B2F_BWD_DEBUG_CLOCK=1): every 512th
    // CTA prints its cycles per phase.  ncu reports this launch at half its stand-alone duration, so this is the
    // instrument for it; compiled out by default (the printf costs registers and stack).
    long long dbg_c0 = 0; unsigned long long dbg_t0 = 0;
    if ((A.flags & 0x200) && threadIdx.x == 0 && (blockIdx.x % 512) == 0) {
        dbg_c0 = clock64();
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(dbg_t0));
    }
#endif
    BTile b;
    Tile& t = b.t;
    t.D = A.D; t.TM = A.TM; t.logTM = A.logTM; t.XS = A.XS; t.HS = A.HS; t.WPG = A.WPG; t.G = A.G; t.flip = 0;
    const int tid = threadIdx.x, NT = blockDim.x, lane = tid & 31, warp = tid >> 5, NW = NT >> 5;
    const int D = A.D, TM = A.TM, XS = A.XS, HS = A.HS;
    t.xt = smem;
    b.gt = t.xt + TM * XS;
    t.hid = b.gt + TM * XS;
    b.dhid = t.hid + TM * HS;
    t.act = b.dhid;                        // scratch of the sequential forward recompute (dhid is idle in phase A)
    t.ldp = b.dhid + TM * HS;              // [WPG][TM] (written by the forward recompute, unused)
    b.GL = t.ldp + A.WPG * TM;             // [TM]
    float* ea = b.GL + TM;                 // [3*D]
    b.dhs = ea + ((3 * D + 3) & ~3);       // [NW][32][dhs_pp], 16-byte aligned
    b.dhp = b.dhs + NW * 32 * A.dhs_pp;    // [WPG][TM][HS]
    b.wst = b.dhp + ((A.WPG * TM * HS + 3) & ~3);
    b.wst_stride = A.wst_stride;
    const long long row0 = (long long)blockIdx.x * TM;
    const int rows = (int)min((long long)TM, A.B - row0);
    b.rows = rows;
    b.precise = A.flags & B2F_FLOW_MODE_PRECISE;

    for (int m = warp; m < TM; m += NW) {
        float* dst = t.xt + m * XS;
        for (int j = lane; j < D; j += 32) dst[j] = (m < rows) ? __ldg(A.x + (row0 + m) * D + j) : 0.0f;
    }
    __syncthreads();

    // ---- phase A: forward recompute, saving the input of every conditioner layer ---------------------
    // (skipped when the forward pass already saved them, B2F_FLOW_WS_FILLED: the tile loaded above is then the flow's
    //  OUTPUT and only the flip state has to be brought to the end of the program)
    if (A.flags & B2F_FLOW_WS_FILLED) {
        for (int oi = 0; oi < A.n_ops; ++oi)
            if (A.ops[oi].f.kind == B2F_OP_FLIP) t.flip ^= 1;
    } else
    for (int oi = 0; oi < A.n_ops; ++oi) {
        const BwdOp& op = A.ops[oi];
        if (op.f.kind == B2F_OP_FLIP) { t.flip ^= 1; continue; }
        if (op.f.kind == B2F_OP_ELEMENTWISE && (op.f.flags & B2F_FLAG_ROW_BIAS)) {
            // context-conditioned elementwise layer: per-row parameters (B, D, 2)
            const float* pr = op.f.p0 + (size_t)row0 * D * 2;
            const bool fwd = op.f.tkind == B2F_T_AFFINE_FWD;
            for (int idx = tid; idx < rows * D; idx += NT) {
                const int m = idx / D, j = idx - m * D, c = t.col(j);
                const float2 u = __ldg(reinterpret_cast<const float2*>(pr + (size_t)idx * 2));
                float a, la;
                affine_scale<0>(u.x, a, la);
                t.xt[m * XS + c] = fwd ? fmaf(a, t.xt[m * XS + c], u.y) : (t.xt[m * XS + c] - u.y) / a;
            }
            __syncthreads();
            continue;
        }
        if (op.f.kind == B2F_OP_ELEMENTWISE) {
            elementwise_stage(ea, op.f, D);
            __syncthreads();
            elementwise_apply(t, ea, op.f.tkind == B2F_T_AFFINE_FWD);
            __syncthreads();
            continue;
        }
        float* save = A.ws + op.ws_off + row0 * D;
        for (int m = warp; m < rows; m += NW)
            for (int j = lane; j < D; j += 32) save[(size_t)m * D + j] = t.xt[m * XS + j];   // physical layout
        if (op.f.kind == B2F_OP_MADE_SEQ) {
            __syncthreads();
            run_sequential_forward<MODE>(t, op.f);
            __syncthreads();
            continue;
        }
        const bool coupling = op.f.kind == B2F_OP_COUPLING;
        const int n_src = coupling ? D / 2 : D, t0 = coupling ? D / 2 : 0;
        hidden_layer<true>(t, op.f, n_src, (op.f.flags & B2F_FLAG_ROW_BIAS) ? op.f.p1 + row0 * op.f.H : nullptr, rows);
        __syncthreads();
        run_transform_forward<MODE>(t, op.f, t0, D - t0);
        __syncthreads();
    }

#ifdef B2F_BWD_CLOCK_HOOK
    long long dbg_cA = 0, dbg_cT = 0, dbg_cH = 0, dbg_cR = 0;
    const bool dbg = (A.flags & 0x200) && threadIdx.x == 0 && (blockIdx.x % 512) == 0;
    if (dbg) dbg_cA = clock64();
#endif
    // ---- gradient seed: dL/dz = gy + glp * d base_logp / dz ;  dL/dlog_det = gld + glp ------------------
    for (int m = warp; m < TM; m += NW) {
        const bool live = m < rows;
        const float glp = (live && A.glp) ? __ldg(A.glp + row0 + m) : 0.0f;
        for (int j = lane; j < D; j += 32) {
            const int c = t.col(j);
            float gseed = (live && A.gy) ? __ldg(A.gy + (row0 + m) * D + j) : 0.0f;
            if (A.glp) {
                const float loc = A.base_loc ? __ldg(A.base_loc + j) : 0.0f;
                const float lsc = A.base_log_scale ? __ldg(A.base_log_scale + j) : 0.0f;
                const float is = expf(-lsc);
                gseed -= glp * (t.xt[m * XS + c] - loc) * is * is;     // d/dz of -(0.5*((z-loc)/scale)^2 + ...)
            }
            b.gt[m * XS + c] = gseed;
        }
        if (lane == 0) b.GL[m] = live ? ((A.gld ? __ldg(A.gld + row0 + m) : 0.0f) + glp) : 0.0f;
    }
    __syncthreads();

    // ---- phase B: reverse walk ---------------------------------------------------------------------------
    for (int oi = A.n_ops - 1; oi >= 0; --oi) {
        const BwdOp& op = A.ops[oi];
        if (op.f.kind == B2F_OP_FLIP) { t.flip ^= 1; continue; }
        if (op.f.kind == B2F_OP_ELEMENTWISE && (op.f.flags & B2F_FLAG_ROW_BIAS)) {
            // per-row parameters: un-do the layer in place, propagate the gradient, WRITE the parameter gradient per row
            const float* pr = op.f.p0 + (size_t)row0 * D * 2;
            const bool fwd = op.f.tkind == B2F_T_AFFINE_FWD;
            for (int idx = tid; idx < rows * D; idx += NT) {
                const int m = idx / D, j = idx - m * D, c = t.col(j);
                const float2 u = __ldg(reinterpret_cast<const float2*>(pr + (size_t)idx * 2));
                float a, la;
                affine_scale<0>(u.x, a, la);
                const float ia = 1.0f / a, zo = t.xt[m * XS + c], gz = b.gt[m * XS + c], GLm = b.GL[m];
                float du0, du1;
                if (fwd) {                     // z = a*x + b, ld += log a
                    const float xi = (zo - u.y) * ia;
                    du0 = gz * xi + GLm * ia;
                    du1 = gz;
                    t.xt[m * XS + c] = xi;
                    b.gt[m * XS + c] = gz * a;
                } else {                       // z = (x - b)/a, ld -= log a
                    du0 = -gz * zo * ia - GLm * ia;
                    du1 = -gz * ia;
                    t.xt[m * XS + c] = fmaf(a, zo, u.y);
                    b.gt[m * XS + c] = gz * ia;
                }
                if (op.g0) {
                    float* gp = op.g0 + ((size_t)row0 * D + idx) * 2;
                    gp[0] = du0 * (a - kAffineM) * 0.5f;
                    gp[1] = du1;
                }
            }
            __syncthreads();
            continue;
        }
        if (op.f.kind == B2F_OP_ELEMENTWISE) {
            elementwise_stage(ea, op.f, D);
            __syncthreads();
            const bool fwd = op.f.tkind == B2F_T_AFFINE_FWD;
            // thread per column: un-do the layer in place, propagate the gradient, reduce the parameter gradient
            for (int j = tid; j < D; j += NT) {
                const int c = t.col(j);
                const float a = ea[j], bta = ea[D + j], ia = 1.0f / a;
                float du0 = 0.0f, du1 = 0.0f;
                for (int m = 0; m < TM; ++m) {
                    const float zo = t.xt[m * XS + c], gz = b.gt[m * XS + c], GLm = b.GL[m];
                    if (fwd) {                     // z = a*x + b, ld += log a
                        const float xi = (zo - bta) * ia;
                        du0 += gz * xi + GLm * ia;
                        du1 += gz;
                        t.xt[m * XS + c] = xi;
                        b.gt[m * XS + c] = gz * a;
                    } else {                       // z = (x - b)/a, ld -= log a
                        du0 += -gz * zo * ia - GLm * ia;
                        du1 += -gz * ia;
                        t.xt[m * XS + c] = fmaf(a, zo, bta);
                        b.gt[m * XS + c] = gz * ia;
                    }
                }
                if (op.g0) {
                    atomicAdd(op.g0 + 2 * j, du0 * (a - kAffineM) * 0.5f);
                    atomicAdd(op.g0 + 2 * j + 1, du1);
                }
            }
            __syncthreads();
            continue;
        }
        const float* saved = A.ws + op.ws_off + row0 * D;
        if (op.f.kind == B2F_OP_MADE_SEQ) {
            // xt holds this layer's OUTPUT x (later layers were un-done); its input z is in the workspace
            run_sequential_backward<MODE>(b, op, saved);
            __syncthreads();
            const int H = op.f.H;
            if (op.g0) {
                for (int idx = tid; idx < H * D; idx += NT) {
                    const int j = idx / D, k = idx - j * D;
                    const int c = t.col(k);
                    float sacc = 0.0f;
                    for (int m = 0; m < TM; ++m) sacc = fmaf(b.dhid[m * HS + j], t.xt[m * XS + c], sacc);
                    atomicAdd(op.g0 + idx, sacc);
                }
                for (int j = tid; j < H; j += NT) {
                    float sacc = 0.0f;
                    for (int m = 0; m < TM; ++m) sacc += b.dhid[m * HS + j];
                    atomicAdd(op.g1 + j, sacc);
                }
            }
            __syncthreads();
            for (int m = warp; m < TM; m += NW)
                for (int j = lane; j < D; j += 32) t.xt[m * XS + j] = (m < rows) ? saved[(size_t)m * D + j] : 0.0f;
            __syncthreads();
            continue;
        }
        // conditioner layer: reload its input, recompute hidden activations
        for (int m = warp; m < TM; m += NW)
            for (int j = lane; j < D; j += 32) t.xt[m * XS + j] = (m < rows) ? saved[(size_t)m * D + j] : 0.0f;
        __syncthreads();
        const bool coupling = op.f.kind == B2F_OP_COUPLING;
        const int n_src = coupling ? D / 2 : D, t0 = coupling ? D / 2 : 0, H = op.f.H;
#ifdef B2F_BWD_CLOCK_HOOK
        long long c_a = 0, c_b = 0, c_c = 0;
        if (dbg) c_a = clock64();
#endif
        hidden_layer<true>(t, op.f, n_src, (op.f.flags & B2F_FLAG_ROW_BIAS) ? op.f.p1 + row0 * op.f.H : nullptr, rows);
        __syncthreads();
#ifdef B2F_BWD_CLOCK_HOOK
        if (dbg) c_b = clock64();
#endif
        run_transform_backward<MODE>(b, op, t0, D - t0);
        __syncthreads();
#ifdef B2F_BWD_CLOCK_HOOK
        if (dbg) { c_c = clock64(); dbg_cH += c_b - c_a; dbg_cT += c_c - c_b; dbg_cR -= c_c; }
#endif
        // tanh': dpre = dhid * (1 - hid^2)
        for (int idx = tid; idx < (H << t.logTM); idx += NT) {
            const int m = idx & (TM - 1), j = idx >> t.logTM;
            const float a = t.hid[m * HS + j];
            float d = 0.0f;
            for (int sl = 0; sl < A.WPG; ++sl) d += b.dhp[((size_t)sl * TM + m) * HS + j];
            b.dhid[m * HS + j] = d * (1.0f - a * a);
        }
        __syncthreads();
        if (op.g0) {
            // dL/dW1[j][k] = sum_m dpre[m][j] * x_src[m][k];  dL/db1[j] = sum_m dpre[m][j]
            for (int idx = tid; idx < H * n_src; idx += NT) {
                const int j = idx / n_src, k = idx - j * n_src;
                const int c = t.col(k);
                float s = 0.0f;
                for (int m = 0; m < TM; ++m) s = fmaf(b.dhid[m * HS + j], t.xt[m * XS + c], s);
                atomicAdd(op.g0 + idx, s);
            }
            if (op.f.flags & B2F_FLAG_ROW_BIAS) {
                // context-conditioned layer: dL/d(pre-activation) per row; the caller owns the chain to b1 / context
                for (int idx = tid; idx < rows * H; idx += NT) {
                    const int m = idx / H, j = idx - m * H;
                    op.g1[(row0 + m) * H + j] = b.dhid[m * HS + j];
                }
            } else {
                for (int j = tid; j < H; j += NT) {
                    float s = 0.0f;
                    for (int m = 0; m < TM; ++m) s += b.dhid[m * HS + j];
                    atomicAdd(op.g1 + j, s);
                }
            }
        }
        // dL/dx_src[m][k] += sum_j dpre[m][j] * W1[j][k]
        for (int idx = tid; idx < (n_src << t.logTM); idx += NT) {
            const int m = idx & (TM - 1), k = idx >> t.logTM;
            float s = 0.0f;
            for (int j = 0; j < H; ++j) s = fmaf(b.dhid[m * HS + j], __ldg(op.f.p0 + (size_t)j * n_src + k), s);
            b.gt[m * XS + t.col(k)] += s;
        }
        __syncthreads();
    }

    if (A.gx) {
        for (int m = warp; m < rows; m += NW)
            for (int j = lane; j < D; j += 32) A.gx[(row0 + m) * D + j] = b.gt[m * XS + t.col(j)];
    }
#ifdef B2F_BWD_CLOCK_HOOK
    if ((A.flags & 0x200) && threadIdx.x == 0 && (blockIdx.x % 512) == 0) {
        unsigned long long t1;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
        const long long c1 = clock64();
        printf("[bwd dbg] block %d: %lld cycles, %llu ns, start at %llu ns; phase A %lld, hidden recompute (B) %lld, transform backward %lld\n",
               blockIdx.x, c1 - dbg_c0, t1 - dbg_t0, dbg_t0, dbg_cA - dbg_c0, dbg_cH, dbg_cT);
    }
#endif
}

static int ilog2b(int v) { int l = 0; while ((1 << l) < v) ++l; return l; }

// Tile shape of the backward kernel for a program: rows per tile TM, threads NT, and whether spline layers stage one
// element's output-layer weights per warp (wst_stride > 0: tensor-core path).  Preferred shapes first, then smaller ones
// (fewer warps, then without the weight staging) until the shared-memory footprint fits; false if nothing fits.
// b2f_flow_backward_fits() answers the same question for callers that must decide before building a program.
struct BwdShape { int TM, NT, wst_stride, dhs_pp; size_t smem; };

// padded parameters per element of the widest transformer of a program: 32 with a linear rational spline, else 24
static int bwd_dhs_pp(const b2f_op_t* ops, int32_t n_ops) {
    for (int i = 0; i < n_ops; ++i)
        if ((ops[i].kind == B2F_OP_COUPLING || ops[i].kind == B2F_OP_MADE || ops[i].kind == B2F_OP_MADE_SEQ) &&
            (ops[i].tkind == B2F_T_LRS_FWD || ops[i].tkind == B2F_T_LRS_INV))
            return 32;
    return 24;
}

static bool bwd_tile_shape(const b2f_op_t* ops, int32_t n_ops, int32_t D, int32_t flags, BwdShape& out) {
    int Hmax = 1, Hrq = 0;
    bool rq_aligned = true;
    for (int i = 0; i < n_ops; ++i) {
        const b2f_op_t& o = ops[i];
        if (o.kind == B2F_OP_COUPLING || o.kind == B2F_OP_MADE || o.kind == B2F_OP_MADE_SEQ) Hmax = std::max(Hmax, o.n_hidden);
        if ((o.kind == B2F_OP_COUPLING || o.kind == B2F_OP_MADE) && (o.tkind == B2F_T_RQ_FWD || o.tkind == B2F_T_RQ_INV) &&
            o.n_hidden <= 31) {
            Hrq = std::max(Hrq, o.n_hidden);
            if (reinterpret_cast<uintptr_t>(o.p[2]) & 15) rq_aligned = false;
        }
    }
    const int XS = D | 1, HS = Hmax | 1, dhs_pp = bwd_dhs_pp(ops, n_ops);
    const int wst_pref = (Hrq > 0 && rq_aligned && !(flags & B2F_FLOW_MODE_PRECISE)) ? ((Hrq * 24 + 24 + 3) & ~3) : 0;
    auto smem_bytes = [&](int tm, int nt, int wst) {
        const int wpg = (nt / 32) / (tm / 32);
        return (size_t)sizeof(float) * (2 * (size_t)tm * XS + 2 * (size_t)tm * HS + (((size_t)wpg * tm * HS + 3) & ~3) +
                                        (size_t)wpg * tm + tm + ((3 * D + 3) & ~3) + (size_t)(nt / 32) * 32 * dhs_pp +
                                        (size_t)(nt / 32) * 2 * wst + 4);
    };
    // spline programs: 12 warps on one 32-row tile (the kernel is latency-bound: measured 10.4 ms against 11.6 ms for
    // 8 warps on 64 rows, CouplingRQNSF-256, 131072 rows); everything else: 8 warps on 64 rows
    struct Try { int tm, nt, wst; };
    Try tries[8];
    int n = 0;
    const char *etm = getenv("B2F_BWD_TM"), *ent = getenv("B2F_BWD_NT");
    if (etm || ent) tries[n++] = {etm ? atoi(etm) : (wst_pref ? 32 : 64), ent ? atoi(ent) : (wst_pref ? 384 : 256), wst_pref};
    if (wst_pref) { tries[n++] = {32, 384, wst_pref}; tries[n++] = {32, 256, wst_pref}; tries[n++] = {32, 128, wst_pref}; }
    tries[n++] = {64, 256, 0}; tries[n++] = {32, 256, 0}; tries[n++] = {32, 128, 0}; tries[n++] = {32, 64, 0};
    for (size_t limit : {(size_t)200 * 1024, (size_t)227 * 1024})       // leave room for a second resident CTA first
        for (int i = 0; i < n; ++i) {
            const int TM = tries[i].tm, NT = tries[i].nt;
            if (TM < 32 || (TM & (TM - 1)) || NT % 32 || NT > 384 || (NT / 32) % (TM / 32) || NT / 32 < TM / 32) continue;
            const size_t smem = smem_bytes(TM, NT, tries[i].wst);
            if (smem > limit) continue;
            out.TM = TM; out.NT = NT; out.wst_stride = tries[i].wst; out.dhs_pp = dhs_pp; out.smem = smem;
            return true;
        }
    return false;
}

}  // namespace b2f

using namespace b2f;

extern "C" int64_t b2f_flow_backward_workspace(const b2f_op_t* ops, int32_t n_ops, int64_t B, int32_t D) {
    int64_t n = 0;
    for (int i = 0; i < n_ops; ++i)
        if (ops[i].kind == B2F_OP_COUPLING || ops[i].kind == B2F_OP_MADE || ops[i].kind == B2F_OP_MADE_SEQ) ++n;
    return n * B * (int64_t)D * (int64_t)sizeof(float);
}

extern "C" int32_t b2f_flow_backward_fits(const b2f_op_t* ops, int32_t n_ops, int32_t D) {
    if (!ops || n_ops < 0 || n_ops > B2F_MAX_OPS || D <= 0) return 0;
    BwdShape shape;
    return bwd_tile_shape(ops, n_ops, D, 0, shape) ? 1 : 0;
}

extern "C" int32_t b2f_flow_backward_shape(const b2f_op_t* ops, int32_t n_ops, int32_t D, int32_t flags, int32_t out[3]) {
    if (!ops || n_ops < 0 || n_ops > B2F_MAX_OPS || D <= 0 || !out) return 0;
    if (getenv("B2F_BWD_NO_MMA")) flags |= B2F_FLOW_MODE_PRECISE;     // as b2f_flow_backward does
    BwdShape shape;
    if (!bwd_tile_shape(ops, n_ops, D, flags, shape)) return 0;
    out[0] = shape.TM; out[1] = shape.NT; out[2] = shape.wst_stride;
    return 1;
}

extern "C" int b2f_flow_backward(const b2f_op_t* ops, int32_t n_ops, const float* x, const float* gy,
                                 const float* glog_det, const float* glog_prob, const float* base_loc,
                                 const float* base_log_scale, float* gx, void* workspace, int64_t B, int32_t D,
                                 int32_t flags, void* stream) {
    if (B == 0 && n_ops >= 0 && D > 0) return B2F_OK;      // empty batch: nothing to do (pointers may be null)
    if (!ops || n_ops < 0 || !x || D <= 0 || B < 0) return fail(B2F_ERR_INVALID, "b2f_flow_backward: bad arguments");
    if (n_ops > B2F_MAX_OPS) return fail(B2F_ERR_UNSUPPORTED, "b2f_flow_backward: %d ops > B2F_MAX_OPS", n_ops);
    if (B == 0) return B2F_OK;
    BwdArgs A;
    memset(&A, 0, sizeof(A));
    int Hmax = 1;
    long long off = 0;
    for (int i = 0; i < n_ops; ++i) {
        const b2f_op_t& o = ops[i];
        BwdOp& d = A.ops[i];
        d.f.kind = o.kind; d.f.tkind = o.tkind; d.f.H = o.n_hidden; d.f.flags = o.flags; d.f.boundary = o.boundary;
        d.f.p0 = (const float*)o.p[0]; d.f.p1 = (const float*)o.p[1]; d.f.p2 = (const float*)o.p[2];
        d.f.p3 = (const float*)o.p[3]; d.f.p4 = nullptr;
        d.g0 = (float*)o.g[0]; d.g1 = (float*)o.g[1]; d.g2 = (float*)o.g[2]; d.g3 = (float*)o.g[3];
        d.ws_off = -1;
        switch (o.kind) {
            case B2F_OP_FLIP: break;
            case B2F_OP_ELEMENTWISE:
                if (!o.p[0]) return fail(B2F_ERR_INVALID, "op %d: elementwise layer without parameters", i);
                if (o.tkind != B2F_T_AFFINE_FWD && o.tkind != B2F_T_AFFINE_INV)
                    return fail(B2F_ERR_UNSUPPORTED, "op %d: elementwise transformer kind %d", i, o.tkind);
                break;
            case B2F_OP_COUPLING: case B2F_OP_MADE: {
                if (!o.p[0] || !o.p[1] || !o.p[2] || !o.p[3] || o.n_hidden <= 0)
                    return fail(B2F_ERR_INVALID, "op %d: conditioner parameters missing", i);
                if ((o.tkind == B2F_T_RQ_FWD || o.tkind == B2F_T_RQ_INV) && o.n_bins != 8)
                    return fail(B2F_ERR_UNSUPPORTED, "op %d: fused RQ spline needs n_bins == 8", i);
                if ((o.tkind == B2F_T_LRS_FWD || o.tkind == B2F_T_LRS_INV) && (o.n_bins != 8 || !(o.boundary > 0.0f)))
                    return fail(B2F_ERR_UNSUPPORTED, "op %d: fused linear rational spline needs n_bins == 8 and a boundary", i);
                if (o.tkind != B2F_T_SHIFT_ADD && o.tkind != B2F_T_SHIFT_SUB && o.tkind != B2F_T_AFFINE_FWD &&
                    o.tkind != B2F_T_AFFINE_INV && o.tkind != B2F_T_RQ_FWD && o.tkind != B2F_T_RQ_INV &&
                    o.tkind != B2F_T_LRS_FWD && o.tkind != B2F_T_LRS_INV)
                    return fail(B2F_ERR_UNSUPPORTED, "op %d: transformer kind %d has no fused backward", i, o.tkind);
                const bool any_g = o.g[0] || o.g[1] || o.g[2] || o.g[3];
                if (any_g && !(o.g[0] && o.g[1] && o.g[2] && o.g[3]))
                    return fail(B2F_ERR_INVALID, "op %d: give all four gradient buffers or none", i);
                if (!workspace) return fail(B2F_ERR_INVALID, "b2f_flow_backward: workspace missing");
                d.ws_off = off;
                off += B * (long long)D;
                Hmax = std::max(Hmax, o.n_hidden);
                break;
            }
            case B2F_OP_MADE_SEQ: {
                if (!o.p[0] || !o.p[1] || !o.p[2] || !o.p[3] || !o.p[4] || o.n_hidden <= 0)
                    return fail(B2F_ERR_INVALID, "op %d: conditioner parameters missing", i);
                const bool rq = o.tkind == B2F_T_RQ_INV || o.tkind == B2F_T_RQ_FWD || o.tkind == B2F_T_LRS_INV ||
                                o.tkind == B2F_T_LRS_FWD;
                if (o.tkind == B2F_T_RQ_FWD || o.tkind == B2F_T_LRS_FWD)
                    return fail(B2F_ERR_UNSUPPORTED, "op %d: sequential forward spline", i);
                if (o.tkind != B2F_T_SHIFT_ADD && o.tkind != B2F_T_SHIFT_SUB && o.tkind != B2F_T_AFFINE_FWD &&
                    o.tkind != B2F_T_AFFINE_INV && !rq)
                    return fail(B2F_ERR_UNSUPPORTED, "op %d: transformer kind %d has no fused backward", i, o.tkind);
                if (o.tkind == B2F_T_LRS_INV && !(o.boundary > 0.0f))
                    return fail(B2F_ERR_UNSUPPORTED, "op %d: linear rational spline needs a boundary", i);
                if (rq && (o.n_bins != 8 || !(o.flags & B2F_FLAG_SEQ_LOGDET_EXACT)))
                    return fail(B2F_ERR_UNSUPPORTED,
                                "op %d: the backward of a sequential spline layer needs B2F_FLAG_SEQ_LOGDET_EXACT (the "
                                "reference's last-iteration log-det has no fused gradient) and n_bins == 8", i);
                const bool any_g = o.g[0] || o.g[1] || o.g[2] || o.g[3];
                if (any_g && !(o.g[0] && o.g[1] && o.g[2] && o.g[3]))
                    return fail(B2F_ERR_INVALID, "op %d: give all four gradient buffers or none", i);
                if (!workspace) return fail(B2F_ERR_INVALID, "b2f_flow_backward: workspace missing");
                d.f.p4 = (const int*)o.p[4];
                d.ws_off = off;
                off += B * (long long)D;
                Hmax = std::max(Hmax, o.n_hidden);
                break;
            }
            default: return fail(B2F_ERR_INVALID, "op %d: unknown kind %d", i, o.kind);
        }
    }
    A.n_ops = n_ops; A.D = D; A.B = B; A.flags = flags;
    A.x = x; A.gy = gy; A.gld = glog_det; A.glp = glog_prob; A.base_loc = base_loc; A.base_log_scale = base_log_scale;
    A.gx = gx; A.ws = (float*)workspace;
    A.XS = D | 1; A.HS = Hmax | 1;
    if (flags & B2F_FLOW_WS_FILLED) {
        int nflip = 0;
        for (int i = 0; i < n_ops; ++i) nflip += ops[i].kind == B2F_OP_FLIP;
        if (nflip & 1) return fail(B2F_ERR_UNSUPPORTED, "b2f_flow_backward: B2F_FLOW_WS_FILLED needs an even number of FLIP ops");
        if (!workspace) return fail(B2F_ERR_INVALID, "b2f_flow_backward: B2F_FLOW_WS_FILLED without a workspace");
    }
    if (getenv("B2F_BWD_NO_MMA")) A.flags |= B2F_FLOW_MODE_PRECISE;
    if (getenv("B2F_BWD_DEBUG_CLOCK")) A.flags |= 0x200;
    BwdShape shape;
    if (!bwd_tile_shape(ops, n_ops, D, A.flags, shape))
        return fail(B2F_ERR_UNSUPPORTED, "b2f_flow_backward: D=%d H=%d does not fit shared memory", D, Hmax);
    A.wst_stride = shape.wst_stride;
    A.dhs_pp = shape.dhs_pp;
    const int TM = shape.TM, NT = shape.NT;
    const size_t smem = shape.smem;
    A.TM = TM; A.logTM = ilog2b(TM); A.G = TM / 32; A.WPG = (NT / 32) / A.G;
    const long long grid = (B + TM - 1) / TM;
    if (grid > 0x7fffffffLL) return fail(B2F_ERR_UNSUPPORTED, "b2f_flow_backward: batch too large for one launch");
    // gradients of the spline knots cancel at the 1e-3 level in fp32 (tests/test_c_oracle_and_hostmath.py): always use the
    // accurate exp / log / division variants here, whatever arithmetic mode the forward pass runs in
    auto kern = flow_backward_kernel<0>;
    cudaError_t ce = (cudaError_t)raise_smem_limit((const void*)kern, smem);
    if (ce != cudaSuccess) return fail(B2F_ERR_CUDA, "cudaFuncSetAttribute: %s", cudaGetErrorString(ce));
    kern<<<(unsigned)grid, NT, smem, (cudaStream_t)stream>>>(A);
    return check_launch("b2f_flow_backward");
}
