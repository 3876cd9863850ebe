// Whole-flow fused kernel, row-per-thread variant (kernel K3) -- device code, instantiated by b2f_flow_rows.cu (affine /
// shift programs) and b2f_flow_rows_rq.cu (programs with sequential spline layers): small conditioners (hidden width <= 32) on the
// FP32 pipe with every per-sample quantity in registers.
//
// Same program, operands and results as the generic kernel in b2f_flow.cu (which stays the fallback for shapes this
// one does not take); replaces the same reference code (file:line relative to /root/reference/torchflows):
//   bijections/base.py:203-232, .../autoregressive/layers_base.py:119-163,202-223,300-318, layers.py:19-69,
//   .../conditioning/transforms.py:197-198,259-264,293-307, matrix/permutation.py:19-37, flows.py:628-648,
//   base_distributions/gaussian.py:46-54.
//
// Why a second mapping: for RealNVP / NICE / MAF / IAF shapes (D <= a few hundred, H ~ 6..17, 1-2 parameters per
// element) the conditioner is ~1-2 kFLOP per row -- far too small for a 128-row tensor-core tile pipeline (measured:
// barrier round trips dominate) and dominated by shared-memory traffic and __syncthreads in the warp-per-element
// mapping of b2f_flow.cu.  Here a THREAD owns R rows for the whole program:
//   * the hidden activations hid[R][HP] and the transformer parameters acc[R][P] live in registers (R = 1 is what ships:
//     two rows per thread measured slower, occupancy beats weight reuse);
//   * the weights of EVERY conditioner layer are staged once per CTA in shared memory, zero-padded to HP = 4*HP4 hidden
//     units with the output bias in a constant-1 hidden slot, so every inner loop has a compile-time trip count and a
//     weight is one broadcast 16-byte shared-memory load that feeds 4 FFMAs in each of the 32 lanes; spline layers (23 x H
//     weights per element) stream the next element's block into a per-warp double buffer with cp.async instead;
//   * a warp only ever touches its own 32 rows (cp.async tile load, several tiles per warp), so after the one staging
//     barrier there is no CTA barrier at all: layers, the D-step sequential inverse of a masked autoregressive layer
//     (layers_base.py:213-223) and the base log-density run back to back, warps drift freely and hide each other's
//     latency;
//   * all-sequential programs that write an output keep their rows in the output buffer itself (`inplace`: a thread walks
//     its own row of y in global memory, L1 holds its current line): no tile, so registers, not shared memory, bound the
//     resident warps;
//   * the tile row stride XS is a multiple of 4 floats with XS/4 odd, so a thread reads/writes 4 consecutive columns
//     of its row with one conflict-free 16-byte shared-memory access;
//   * ReversePermutationMatrix (matrix/permutation.py:19-37) never moves data: a FLIP only toggles how logical columns
//     map to physical ones, and that mapping is folded into the WEIGHT staging (the staged images are indexed by
//     physical column), so every inner loop walks physical columns upwards with constant offsets;
//   * a run of elementwise layers (ElementwiseAffine / ActNorm) is one affine map per column that the next conditioner
//     layer, or the epilogue, applies to the values it loads anyway.
// HBM traffic is the algorithmic minimum (x read once, z / log-density written once, weights from L1/L2).
#pragma once
#include "b2f_flow_device.cuh"
#include "b2f_rqfast.cuh"

namespace b2f {

// CTA size: four warps for affine / shift programs, two for programs with sequential spline layers (their larger
// register footprint and per-warp staging buffers pack better in small CTAs); warps run independently after the one
// staging barrier, so the CTA size only sets how many warps share one copy of the weights.

struct RowsArgs {
    DevOp ops[B2F_MAX_OPS];
    int n_ops, D, XS, flags, n_runs, tiles_per_warp;
    int wtotal, rq_stride;      // floats of all staged weights; floats per per-warp streaming buffer (spline layers)
    int inplace;                // spline programs with an output buffer: rows live in y (global memory), no shared tile
    int woff[B2F_MAX_OPS];      // float offset of each conditioner layer's staged weights in the weight area
    long long B;
    const float* x;
    float* y;
    float* log_det;
    float* log_prob;
    const float* base_loc;
    const float* base_log_scale;
};

// 4 consecutive PHYSICAL columns c0..c0+3 of a row (c0 % 4 == 0)
__device__ __forceinline__ void ld4(const float* xr, int c0, float (&v)[4]) {
    const float4 q = *reinterpret_cast<const float4*>(xr + c0);
    v[0] = q.x; v[1] = q.y; v[2] = q.z; v[3] = q.w;
}
__device__ __forceinline__ void st4(float* xr, int c0, const float (&v)[4]) {
    *reinterpret_cast<float4*>(xr + c0) = make_float4(v[0], v[1], v[2], v[3]);
}
// z = A_c * x + B_c with the coefficients of a pending elementwise run (er[0..D) = A, er[D..2D) = B, physical columns)
__device__ __forceinline__ void apply_run(const float* er, int D, int c0, float (&v)[4]) {
    float a[4], b[4];
    ld4(er, c0, a);
    ld4(er + D, c0, b);
#pragma unroll
    for (int u = 0; u < 4; ++u) v[u] = fmaf(a[u], v[u], b[u]);
}

// tanh for the hidden layer.  MODE 0: libm-grade tanhf.  MODE >= 1: 1 - 2/(exp(2x)+1) on the SFU (ex2.approx, rcp.approx):
// ABSOLUTE error <= ~2e-7, i.e. the size of one rounding of an activation near 1 -- the activations only feed dot products
// with O(1) weights, so this is rounding-level noise for the transformer parameters (no bin decisions on this path).
template <int MODE> __device__ __forceinline__ float rows_tanh(float x) {
    if constexpr (MODE == 0) return tanhf(x);
    else {
        const float e = exp2f(fminf(x, 44.0f) * 2.885390081777927f);      // exp(2x), clamped below fp32 overflow
        return 1.0f - __fdividef(2.0f, e + 1.0f);
    }
}

// Shared-memory image of one conditioner layer's weights, indexed by PHYSICAL column and zero-padded from H to HP = 4*HP4
// hidden units, so that every inner loop has a compile-time trip count and every weight access is one broadcast 16-byte
// load at a constant offset.  With f = tile currently flipped, physical source column ps0 + kp holds logical source
// k = f ? n_src-1-kp : kp and physical target column pt0 + ep holds logical target e = f ? n_tgt-1-ep : ep.
//   w1  [n_src/4][HP][4]   w1[(kp/4)*HP*4 + j*4 + kp%4] = W1[j][k(kp)]        (one-pass layers)
//   w1c [D][HP]            w1c[c*HP + j]                = W1[j][i(c)]         (sequential layers: rank-1 update of step i)
//   b1  [HP]
//   w2  [n_tgt*P][HP]      w2[(ep*P + p)*HP + j]        = W2tile[e(ep)][j][p] for j < H,  b2[e][p] for j == H  (HP > H:
//                          the kernel keeps a constant 1 in hidden slot H, so the bias costs no extra load)
template <int HP>
struct RowsWeights {
    const float *w1, *b1, *w2;
};

template <int HP>
__device__ __forceinline__ RowsWeights<HP> weights_view(const float* wbuf, int n_src) {
    return RowsWeights<HP>{wbuf, wbuf + n_src * HP, wbuf + n_src * HP + HP};
}

template <int HP, int P, int NT>
__device__ __forceinline__ void stage_weights(float* wbuf, const DevOp& op, int n_src, int n_tgt, bool seq, int f) {
    constexpr int kRowsThreads = NT;
    const int H = op.H, tid = threadIdx.x;
    float* w1 = wbuf;
    float* b1 = w1 + n_src * HP;
    float* w2 = b1 + HP;
    if (!seq) {
        for (int d = tid; d < n_src * HP; d += kRowsThreads) {
            const int k4 = d / (HP * 4), rem = d - k4 * (HP * 4), j = rem >> 2, kp = 4 * k4 + (rem & 3);
            const int k = f ? n_src - 1 - kp : kp;
            w1[d] = (j < H) ? __ldg(op.p0 + (size_t)j * n_src + k) : 0.0f;
        }
    } else {
        for (int d = tid; d < n_src * HP; d += kRowsThreads) {
            const int c = d / HP, j = d - c * HP, i = f ? n_src - 1 - c : c;
            w1[d] = (j < H) ? __ldg(op.p0 + (size_t)j * n_src + i) : 0.0f;
        }
    }
    if (tid < HP) b1[tid] = (tid < H) ? __ldg(op.p1 + tid) : 0.0f;
    if constexpr (P > 2) return;        // spline layers: the output layer (P x H per element) is streamed per element
    for (int d = tid; d < n_tgt * P * HP; d += kRowsThreads) {
        const int q = d / HP, j = d - q * HP, ep = q / P, p = q - ep * P;
        const int e = f ? n_tgt - 1 - ep : ep;
        w2[d] = (j < H) ? __ldg(op.p2 + ((size_t)e * H + j) * P + p) : (j == H ? __ldg(op.p3 + e * P + p) : 0.0f);
    }
}

// acc[r][p] = sum_j W2[e][p][j] * hid[r][j]  with the bias in slot H   (transforms.py:297-300, last Linear)
template <int P, int HP, int R>
__device__ __forceinline__ void row_params(float (&acc)[R][P], const float4* __restrict__ w2e, const float (&hid)[R][HP]) {
#pragma unroll
    for (int p = 0; p < P; ++p) {
        float a[R];
#pragma unroll
        for (int r = 0; r < R; ++r) a[r] = 0.0f;
#pragma unroll
        for (int j4 = 0; j4 < HP / 4; ++j4) {
            const float4 w = w2e[p * (HP / 4) + j4];
#pragma unroll
            for (int r = 0; r < R; ++r) {
                a[r] = fmaf(w.x, hid[r][4 * j4 + 0], a[r]);
                a[r] = fmaf(w.y, hid[r][4 * j4 + 1], a[r]);
                a[r] = fmaf(w.z, hid[r][4 * j4 + 2], a[r]);
                a[r] = fmaf(w.w, hid[r][4 * j4 + 3], a[r]);
            }
        }
#pragma unroll
        for (int r = 0; r < R; ++r) acc[r][p] = a[r];
    }
}

// one-pass conditioner layer (coupling, or masked autoregressive in its parallel direction); sources are the physical
// columns [ps0, ps0+n_src), targets [pt0, pt0+n_tgt)
template <int TK, int MODE, int HP, int R>
__device__ __forceinline__ void rows_pass(float* x0, int XS, int D, const DevOp& op, const RowsWeights<HP>& W, int ps0,
                                          int n_src, int pt0, int n_tgt, const float* er, float (&ld)[R],
                                          const float* xin, bool live) {
    // xin / live: in-place mode (rows in global memory), see rows_sequential_rq; xin == nullptr and live == true otherwise
    const float* sin = xin ? xin : x0;
    constexpr int P = TInfo<TK>::P;
    const int H = op.H;
    float hid[R][HP];
#pragma unroll
    for (int j = 0; j < HP; ++j) {
        const float b = W.b1[j];
#pragma unroll
        for (int r = 0; r < R; ++r) hid[r][j] = b;
    }
    // hid[r][j] = tanh(b1[j] + sum_k W1[j][k] x[r][k])                 (transforms.py:295-296 / :259-262)
    const float4* w1 = reinterpret_cast<const float4*>(W.w1);
    for (int c0 = ps0; c0 < ps0 + n_src; c0 += 4, w1 += HP) {
        float xv[R][4];
#pragma unroll
        for (int r = 0; r < R; ++r) {
            xv[r][0] = xv[r][1] = xv[r][2] = xv[r][3] = 0.0f;
            if (live) ld4(sin + r * 32 * XS, c0, xv[r]);
            if (er) apply_run(er, D, c0, xv[r]);   // pending elementwise run: applied to the source columns on the way in
            if ((er || xin) && live) st4(x0 + r * 32 * XS, c0, xv[r]);      // ... and written back (or copied x -> y)
        }
#pragma unroll
        for (int j = 0; j < HP; ++j) {
            const float4 w = w1[j];
#pragma unroll
            for (int r = 0; r < R; ++r) {
                hid[r][j] = fmaf(w.x, xv[r][0], hid[r][j]);
                hid[r][j] = fmaf(w.y, xv[r][1], hid[r][j]);
                hid[r][j] = fmaf(w.z, xv[r][2], hid[r][j]);
                hid[r][j] = fmaf(w.w, xv[r][3], hid[r][j]);
            }
        }
    }
#pragma unroll
    for (int j = 0; j < HP; ++j) {
#pragma unroll
        for (int r = 0; r < R; ++r) hid[r][j] = (j == H) ? 1.0f : rows_tanh<MODE>(hid[r][j]);   // slot H carries the bias;
    }                                                                    // padded units: tanh(0) = 0 times zero weights
    const bool ew_targets = er != nullptr && pt0 != ps0;     // coupling: the loop above did not touch the targets
    const float* tin = (xin && pt0 != ps0) ? xin : x0;       // ... so in-place mode still finds them in the input
    const float4* w2 = reinterpret_cast<const float4*>(W.w2);
    for (int c0 = pt0; c0 < pt0 + n_tgt; c0 += 4, w2 += 4 * P * (HP / 4)) {
        float xv[R][4];
#pragma unroll
        for (int r = 0; r < R; ++r) {
            xv[r][0] = xv[r][1] = xv[r][2] = xv[r][3] = 0.0f;
            if (live) ld4(tin + r * 32 * XS, c0, xv[r]);
            if (ew_targets) apply_run(er, D, c0, xv[r]);
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            float acc[R][P];
            row_params<P, HP, R>(acc, w2 + u * P * (HP / 4), hid);
#pragma unroll
            for (int r = 0; r < R; ++r) {
                float out, l;
                transform_element<TK, MODE, P>(xv[r][u], acc[r], op.boundary, out, l);
                xv[r][u] = out;
                ld[r] += l;
            }
        }
#pragma unroll
        for (int r = 0; r < R; ++r)
            if (live) st4(x0 + r * 32 * XS, c0, xv[r]);
    }
}

// D-step sequential direction of a masked autoregressive layer (layers_base.py:213-223) at the cost of ONE conditioner
// pass: the hidden pre-activations get a rank-1 update per finished dimension and only the P parameters of dimension i
// are evaluated at step i.  Everything of a sample is in its thread's registers: no barrier in the D-step loop.
// REV: the tile is flipped, logical step i lives at physical column D-1-i, so physical columns are walked downwards.
template <int TK, int MODE, int HP, int R, bool REV>
__device__ __forceinline__ void rows_sequential(float* x0, int XS, int D, const DevOp& op, const RowsWeights<HP>& W,
                                                const float* er, float (&ld)[R], const float* xin, bool live) {
    const float* sin = xin ? xin : x0;
    constexpr int P = TInfo<TK>::P;
    const int H = op.H;
    float pre[R][HP], act[R][HP];
    int fin[HP];
#pragma unroll
    for (int j = 0; j < HP; ++j) {
        const float b = W.b1[j];
        fin[j] = (j < H) ? __ldg(op.p4 + j) : -1;
#pragma unroll
        for (int r = 0; r < R; ++r) { pre[r][j] = b; act[r][j] = (j == H) ? 1.0f : 0.0f; }   // slot H carries the bias
    }
    const float4* w1c = reinterpret_cast<const float4*>(W.w1);
    const float4* w2 = reinterpret_cast<const float4*>(W.w2);
    for (int q = 0; q < D; q += 4) {
        const int c0 = REV ? D - 4 - q : q;
        float xv[R][4];
#pragma unroll
        for (int r = 0; r < R; ++r) {
            xv[r][0] = xv[r][1] = xv[r][2] = xv[r][3] = 0.0f;
            if (live) ld4(sin + r * 32 * XS, c0, xv[r]);
            if (er) apply_run(er, D, c0, xv[r]);
        }
#pragma unroll
        for (int uu = 0; uu < 4; ++uu) {
            const int u = REV ? 3 - uu : uu;          // compile-time after unrolling
            const int c = c0 + u, i = q + uu;         // physical column, logical step
            // hidden units whose inputs x_0..x_{i-1} are now all final
#pragma unroll
            for (int j = 0; j < HP; ++j)
                if (fin[j] == i) {
#pragma unroll
                    for (int r = 0; r < R; ++r) act[r][j] = rows_tanh<MODE>(pre[r][j]);
                }
            float acc[R][P];
            row_params<P, HP, R>(acc, w2 + (size_t)c * P * (HP / 4), act);
#pragma unroll
            for (int r = 0; r < R; ++r) {
                float out, l;
                transform_element<TK, MODE, P>(xv[r][u], acc[r], op.boundary, out, l);
                xv[r][u] = out;
                ld[r] += l;
            }
#pragma unroll
            for (int j4 = 0; j4 < HP / 4; ++j4) {
                const float4 w = w1c[c * (HP / 4) + j4];          // column i of the (masked) first layer
#pragma unroll
                for (int r = 0; r < R; ++r) {
                    pre[r][4 * j4 + 0] = fmaf(w.x, xv[r][u], pre[r][4 * j4 + 0]);
                    pre[r][4 * j4 + 1] = fmaf(w.y, xv[r][u], pre[r][4 * j4 + 1]);
                    pre[r][4 * j4 + 2] = fmaf(w.z, xv[r][u], pre[r][4 * j4 + 2]);
                    pre[r][4 * j4 + 3] = fmaf(w.w, xv[r][u], pre[r][4 * j4 + 3]);
                }
            }
        }
#pragma unroll
        for (int r = 0; r < R; ++r)
            if (live) st4(x0 + r * 32 * XS, c0, xv[r]);
    }
}

// The same D-step sequential direction for a SPLINE masked autoregressive layer (MaskedAutoregressiveRQNSF /
// MaskedAutoregressiveLRS sampling, InverseAutoregressiveRQNSF / InverseAutoregressiveLRS density).  The output layer is
// P x H weights PER ELEMENT (tile layout [e][j][PP] in global memory; P = 23, PP = 24 for the rational-quadratic spline,
// P = PP = 32 for the linear rational one): too large to stage for all D elements, so every warp streams the next element's
// block (H*PP + P floats) into its own double buffer with cp.async while it works on the current element.
// `xin`: where this layer reads its input row from (the kernel's input x for the first layer of an in-place program,
// otherwise x0 itself); `live`: the thread owns a real row (threads past the end of the batch still take part in the
// warp-wide weight staging but must not touch global memory).
template <int TK, int MODE, int HP>
__device__ __forceinline__ void rows_sequential_rq(float* x0, const float* xin, bool live, int D, int rev, const DevOp& op,
                                                   const RowsWeights<HP>& W, const float* er, float* wst, int wst_stride,
                                                   float& ld) {
    constexpr int P = TInfo<TK>::P, PP = TInfo<TK>::PP;
    constexpr bool LRS = TK == B2F_T_LRS_FWD || TK == B2F_T_LRS_INV;
    const int H = op.H, lane = threadIdx.x & 31;
    float pre[HP], act[HP];
    int fin[HP];
#pragma unroll
    for (int j = 0; j < HP; ++j) {
        pre[j] = W.b1[j];
        act[j] = 0.0f;
        fin[j] = (j < H) ? __ldg(op.p4 + j) : -1;
    }
    const bool quirk = !(op.flags & B2F_FLAG_SEQ_LOGDET_EXACT);
    // B2F_FLAG_SEQ_FOLDED: p[2] / p[3] hold the FOLDED output layer (24 columns per element, csrc/b2f_rqfast.cuh) and the
    // spline runs in the folded formulation of the tensor-core kernels: ~1/3 of the instructions of the stand-alone one
    const bool folded = !LRS && MODE != 0 && (op.flags & B2F_FLAG_SEQ_FOLDED);
    const float4* w1c = reinterpret_cast<const float4*>(W.w1);
    float* buf[2] = {wst, wst + wst_stride};
    auto stage = [&](int i, float* dst) {            // logical element i
        const float4* src = reinterpret_cast<const float4*>(op.p2 + (size_t)i * H * PP);
        for (int q = lane; q < H * (PP / 4); q += 32) {
            const unsigned d = (unsigned)__cvta_generic_to_shared(dst + 4 * q);
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d), "l"(src + q) : "memory");
        }
        if (lane < (folded ? PP : P)) {
            const unsigned d = (unsigned)__cvta_generic_to_shared(dst + H * PP + lane);
            asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(d), "l"(op.p3 + (size_t)i * (folded ? PP : P) + lane) : "memory");
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    };
    __syncwarp();
    stage(0, buf[0]);
    const bool vec = (D & 3) == 0 && ((reinterpret_cast<uintptr_t>(x0) | reinterpret_cast<uintptr_t>(xin)) & 15) == 0;
    float4 vin = make_float4(0.f, 0.f, 0.f, 0.f), vout = vin;
    // one element per iteration, NOT unrolled: the body holds two inlined spline evaluations (the second one for the
    // reference's log-det quirk) and must stay inside the instruction cache
#pragma unroll 1
    for (int i = 0; i < D; ++i) {
        const int c = rev ? D - 1 - i : i, cur = i & 1;       // physical column of logical step i (rev: flipped tile)
        asm volatile("cp.async.wait_group 0;" ::: "memory");
        __syncwarp();                                 // element i's weights have landed; the other buffer is free
        if (i + 1 < D) stage(i + 1, buf[cur ^ 1]);
        const float* w2e = buf[cur];
        float v;
        if (vec) {
            // four columns per memory access: a thread walks its own row, so a scalar access costs the warp 32 wavefronts per
            // ELEMENT (LSU wavefronts were 72 % busy, profiles/r2_rows_seq_ncu_summary.txt); the group is consumed by rotation
            if ((i & 3) == 0) vin = live ? *reinterpret_cast<const float4*>(xin + (rev ? c - 3 : c)) : make_float4(0.f, 0.f, 0.f, 0.f);
            if (rev) { v = vin.w; vin = make_float4(0.0f, vin.x, vin.y, vin.z); }
            else { v = vin.x; vin = make_float4(vin.y, vin.z, vin.w, 0.0f); }
        } else {
            v = live ? xin[c] : 0.0f;
        }
        if (er) v = fmaf(er[c], v, er[D + c]);
#pragma unroll
        for (int j = 0; j < HP; ++j)
            if (fin[j] == i) act[j] = rows_tanh<MODE>(pre[j]);
        float acc[PP];
#pragma unroll
        for (int p = 0; p < PP; ++p) acc[p] = (p < P || folded) ? w2e[H * PP + p] : 0.0f;
#pragma unroll
        for (int j = 0; j < HP; ++j)
            if (j < H) {
#pragma unroll
                for (int cc = 0; cc < PP / 4; ++cc) {
                    const float4 w = *reinterpret_cast<const float4*>(w2e + j * PP + 4 * cc);
                    acc[4 * cc + 0] = fmaf(w.x, act[j], acc[4 * cc + 0]);
                    acc[4 * cc + 1] = fmaf(w.y, act[j], acc[4 * cc + 1]);
                    acc[4 * cc + 2] = fmaf(w.z, act[j], acc[4 * cc + 2]);
                    acc[4 * cc + 3] = fmaf(w.w, act[j], acc[4 * cc + 3]);
                }
            }
        float out, l;
        if constexpr (LRS) {
            transform_element<TK, MODE, PP>(v, acc, op.boundary, out, l);
            if (quirk && i < D - 1) {
                // the reference's last-iteration log-det (see below): the spline's log-det at the already inverted value
                float out2;
                transform_element<TK, MODE, PP>(out, acc, op.boundary, out2, l);
            }
        } else if (MODE != 0 && folded) {
            constexpr bool INV = TK == B2F_T_RQ_INV;
            if (quirk && i < D - 1) rqf::sequential_step<INV, true, true, (MODE >= 2)>(v, acc, op.boundary, out, l);
            else rqf::sequential_step<INV, true, false, (MODE >= 2)>(v, acc, op.boundary, out, l);
            l *= rqf::kLn2;
        } else if (quirk && i < D - 1) {
            // the reference returns the log-det of its LAST full pass, in which dimension i < D-1 is fed the already
            // inverted value (layers_base.py:218-223, SURVEY Appendix B.3): reproduce that term
            auto h = [&](int q) { return acc[q]; };
            rq_apply_then_logdet_at_output<8, TK == B2F_T_RQ_INV, MODE>(v, h, 8, op.boundary, out, l);
        } else {
            transform_element<TK, MODE, PP>(v, acc, op.boundary, out, l);
        }
        if (vec) {
            if (rev) vout = make_float4(out, vout.x, vout.y, vout.z);
            else vout = make_float4(vout.y, vout.z, vout.w, out);
            if ((i & 3) == 3 && live) *reinterpret_cast<float4*>(x0 + (rev ? c : c - 3)) = vout;
        } else if (live) {
            x0[c] = out;
        }
        ld += l;
#pragma unroll
        for (int j4 = 0; j4 < HP / 4; ++j4) {
            const float4 w = w1c[c * (HP / 4) + j4];              // column i of the (masked) first layer
            pre[4 * j4 + 0] = fmaf(w.x, out, pre[4 * j4 + 0]);
            pre[4 * j4 + 1] = fmaf(w.y, out, pre[4 * j4 + 1]);
            pre[4 * j4 + 2] = fmaf(w.z, out, pre[4 * j4 + 2]);
            pre[4 * j4 + 3] = fmaf(w.w, out, pre[4 * j4 + 3]);
        }
    }
}

template <int TK, int MODE, int HP, int R>
__device__ __forceinline__ void rows_layer_tk(const float* wbuf, float* x0, int XS, int D, int flip, const DevOp& op,
                                              const float* er, float (&ld)[R], const float* xin, bool live) {
    const bool seq = op.kind == B2F_OP_MADE_SEQ;
    const bool coupling = op.kind == B2F_OP_COUPLING;
    const int n_src = coupling ? D / 2 : D, n_tgt = coupling ? D - D / 2 : D;      // HalfSplit: first D//2 logical columns
    const int ps0 = flip ? D - n_src : 0, pt0 = (flip || !coupling) ? 0 : D - n_tgt;
    const RowsWeights<HP> W = weights_view<HP>(wbuf, n_src);
    if (!seq) rows_pass<TK, MODE, HP, R>(x0, XS, D, op, W, ps0, n_src, pt0, n_tgt, er, ld, xin, live);
    else if (flip) rows_sequential<TK, MODE, HP, R, true>(x0, XS, D, op, W, er, ld, xin, live);
    else rows_sequential<TK, MODE, HP, R, false>(x0, XS, D, op, W, er, ld, xin, live);
}

template <int MODE, int HP, int R, bool RQ>
__device__ __forceinline__ void rows_layer(const float* wbuf, float* x0, int XS, int D, int flip, const DevOp& op,
                                           const float* er, float (&ld)[R], float* wst, int wst_stride,
                                           const float* xin = nullptr, bool live = true) {
    if constexpr (RQ) {
        static_assert(R == 1, "spline layers: one row per thread");
        if (op.tkind == B2F_T_RQ_FWD || op.tkind == B2F_T_RQ_INV || op.tkind == B2F_T_LRS_INV) {
            // sequential spline layer (host guarantees MADE_SEQ; linear rational splines: inverse direction only)
            const RowsWeights<HP> W = weights_view<HP>(wbuf, D);
            const float* in = xin ? xin : x0;
            if (op.tkind == B2F_T_RQ_INV) rows_sequential_rq<B2F_T_RQ_INV, MODE, HP>(x0, in, live, D, flip, op, W, er, wst, wst_stride, ld[0]);
            else if (op.tkind == B2F_T_LRS_INV) rows_sequential_rq<B2F_T_LRS_INV, MODE, HP>(x0, in, live, D, flip, op, W, er, wst, wst_stride, ld[0]);
            else rows_sequential_rq<B2F_T_RQ_FWD, MODE, HP>(x0, in, live, D, flip, op, W, er, wst, wst_stride, ld[0]);
            return;
        }
    }
    switch (op.tkind) {
        case B2F_T_SHIFT_ADD: rows_layer_tk<B2F_T_SHIFT_ADD, MODE, HP, R>(wbuf, x0, XS, D, flip, op, er, ld, xin, live); break;
        case B2F_T_SHIFT_SUB: rows_layer_tk<B2F_T_SHIFT_SUB, MODE, HP, R>(wbuf, x0, XS, D, flip, op, er, ld, xin, live); break;
        case B2F_T_AFFINE_FWD: rows_layer_tk<B2F_T_AFFINE_FWD, MODE, HP, R>(wbuf, x0, XS, D, flip, op, er, ld, xin, live); break;
        case B2F_T_AFFINE_INV: rows_layer_tk<B2F_T_AFFINE_INV, MODE, HP, R>(wbuf, x0, XS, D, flip, op, er, ld, xin, live); break;
        default: break;
    }
}

template <int MODE, int HP4, int R, bool RQ, int NT>
__global__ void __launch_bounds__(NT) flow_rows_kernel(const __grid_constant__ RowsArgs A) {
    extern __shared__ __align__(16) float smem[];
    constexpr int kRowsThreads = NT;
    constexpr int NW = kRowsThreads / 32, TMW = 32 * R, HP = 4 * HP4;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int D = A.D, XS = A.XS, D4 = D >> 2;
    float* xw = smem + (size_t)warp * TMW * XS;          // this warp's [32*R][XS] rows
    float* ea = smem + (size_t)NW * TMW * XS;            // [n_runs][2][D]  A_c, B_c of every elementwise run (physical c)
    float* gb = ea + (size_t)A.n_runs * 2 * D;           // [2][D]          base loc_c, 1/scale_c             (physical c)
    float* red = gb + 2 * D;                             // [2][NW]         CTA-uniform constants (partials per warp)
    float* wbuf = red + 2 * NW;                          // staged weights of every conditioner layer (A.woff)
    float* wst = wbuf + A.wtotal + (size_t)warp * 2 * A.rq_stride;   // spline: this warp's double buffer

    // ---- batch-independent part: every run of consecutive elementwise layers is one affine map per column, stored by
    //      the PHYSICAL column it applies to (the flip state at the run is known from the program) -----------------------
    int final_flip = 0;
    {
        float lsum = 0.0f, gsum = 0.0f;
        int run = 0, f = 0;
        for (int oi = 0; oi < A.n_ops; ++oi) {
            if (A.ops[oi].kind == B2F_OP_FLIP) { f ^= 1; continue; }
            if (A.ops[oi].kind != B2F_OP_ELEMENTWISE) continue;
            int n_run = 1;
            while (oi + n_run < A.n_ops && A.ops[oi + n_run].kind == B2F_OP_ELEMENTWISE) ++n_run;
            float* er = ea + (size_t)run * 2 * D;
            for (int c = tid; c < D; c += kRowsThreads) {
                const int j = f ? D - 1 - c : c;
                float Aj = 1.0f, Bj = 0.0f;
                for (int r = 0; r < n_run; ++r) {
                    const DevOp& o = A.ops[oi + r];
                    float a, la;
                    affine_scale<0>(__ldg(o.p0 + 2 * j), a, la);
                    const float b = __ldg(o.p0 + 2 * j + 1);
                    if (o.tkind == B2F_T_AFFINE_FWD) { Aj *= a; Bj = fmaf(a, Bj, b); lsum += la; }
                    else { const float ia = 1.0f / a; Aj *= ia; Bj = (Bj - b) * ia; lsum -= la; }
                }
                er[c] = Aj; er[D + c] = Bj;
            }
            oi += n_run - 1;
            ++run;
        }
        final_flip = f;
        if (A.log_prob) {
            const int gf = (A.flags & B2F_FLOW_LOGP_OF_INPUT) ? 0 : final_flip;      // orientation when the density is taken
            for (int c = tid; c < D; c += kRowsThreads) {
                const int j = gf ? D - 1 - c : c;
                const float lsc = A.base_log_scale ? __ldg(A.base_log_scale + j) : 0.0f;
                gb[c] = A.base_loc ? __ldg(A.base_loc + j) : 0.0f;
                gb[D + c] = expf(-lsc);
                gsum += 0.91893853320467274178f + lsc;
            }
        }
        lsum = warp_sum(lsum);
        gsum = warp_sum(gsum);
        if (lane == 0) { red[warp] = lsum; red[NW + warp] = gsum; }
    }
    // ---- the weights of EVERY conditioner layer, staged once per CTA (physical-column images, see RowsWeights) ---------
    {
        int f = 0;
        for (int oi = 0; oi < A.n_ops; ++oi) {
            const DevOp& op = A.ops[oi];
            if (op.kind == B2F_OP_FLIP) { f ^= 1; continue; }
            if (op.kind == B2F_OP_ELEMENTWISE) continue;
            const bool coupling = op.kind == B2F_OP_COUPLING, seq = op.kind == B2F_OP_MADE_SEQ;
            const int n_src = coupling ? D / 2 : D, n_tgt = coupling ? D - D / 2 : D;
            if (op.tkind == B2F_T_SHIFT_ADD || op.tkind == B2F_T_SHIFT_SUB) stage_weights<HP, 1, NT>(wbuf + A.woff[oi], op, n_src, n_tgt, seq, f);
            else if (op.tkind == B2F_T_RQ_FWD || op.tkind == B2F_T_RQ_INV) stage_weights<HP, 23, NT>(wbuf + A.woff[oi], op, n_src, n_tgt, seq, f);
            else if (op.tkind == B2F_T_LRS_INV) stage_weights<HP, 32, NT>(wbuf + A.woff[oi], op, n_src, n_tgt, seq, f);
            else stage_weights<HP, 2, NT>(wbuf + A.woff[oi], op, n_src, n_tgt, seq, f);
        }
    }
    __syncthreads();   // the only CTA barrier: staged constants and weights visible; from here on warps run independently
    float ldc = 0.0f, gconst = 0.0f;
#pragma unroll
    for (int w = 0; w < NW; ++w) { ldc += red[w]; gconst += red[NW + w]; }
    const bool want_lp = A.log_prob != nullptr;
    float* x0 = xw + lane * XS;                          // row r of this thread: x0 + r*32*XS
    const bool inplace = A.inplace != 0;                 // rows stay in global memory (y): no tile, more resident warps

  for (int tt = 0; tt < A.tiles_per_warp; ++tt) {
    // ---- this warp's next 32*R rows: asynchronous 16-byte copies global -> shared (rows beyond B are zero-filled) -------
    const long long wrow0 = (((long long)blockIdx.x * NW + warp) * A.tiles_per_warp + tt) * TMW;
    const int rows = (int)max(0LL, min((long long)TMW, A.B - wrow0));
    if (rows == 0) break;
    __syncwarp();      // every lane is done with the previous tile
    const bool live = !inplace || lane < rows;
    const float* xin = nullptr;                          // in-place mode: the first layer reads the thread's row of x
    if (inplace) {
        x0 = A.y + (wrow0 + (live ? lane : 0)) * D;
        xin = A.x + (wrow0 + (live ? lane : 0)) * D;
    } else {
        const float4* src = reinterpret_cast<const float4*>(A.x + wrow0 * D);
        int m = 0, c4 = lane;
        while (c4 >= D4) { c4 -= D4; ++m; }
        for (int idx = lane; m < TMW; idx += 32) {
            const unsigned dst = (unsigned)__cvta_generic_to_shared(xw + m * XS + 4 * c4);
            const int nbytes = (m < rows) ? 16 : 0;                     // src-size 0: the 16 bytes are zero-filled
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src + (m < rows ? idx : 0)), "r"(nbytes)
                         : "memory");
            c4 += 32;
            while (c4 >= D4) { c4 -= D4; ++m; }
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
        asm volatile("cp.async.wait_group 0;" ::: "memory");
    }
    __syncwarp();      // the other lanes' copies are visible
    float ld[R], lp[R];
#pragma unroll
    for (int r = 0; r < R; ++r) { ld[r] = 0.0f; lp[r] = 0.0f; }
    const float* er = nullptr;      // elementwise run that has been reached but not applied yet: the next conditioner layer
                                    // (or the epilogue) applies it on the fly to the values it loads anyway
    // DiagonalGaussian.log_prob (gaussian.py:46-54) of the thread's rows as they stand (after the pending run, if any)
    auto base_logp = [&](const float* rowp, bool write_back) {
        float s[R];
#pragma unroll
        for (int r = 0; r < R; ++r) s[r] = 0.0f;
        for (int c0 = 0; c0 < D; c0 += 4) {
            float loc[4], isc[4];
            ld4(gb, c0, loc);
            ld4(gb + D, c0, isc);
#pragma unroll
            for (int r = 0; r < R; ++r) {
                float xv[4] = {0.0f, 0.0f, 0.0f, 0.0f};
                if (live) ld4(rowp + r * 32 * XS, c0, xv);
                if (er) apply_run(er, D, c0, xv);
                if (write_back && live) st4(x0 + r * 32 * XS, c0, xv);       // in-place mode: the trailing elementwise run
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const float t = (xv[u] - loc[u]) * isc[u];
                    s[r] = fmaf(0.5f * t, t, s[r]);
                }
            }
        }
#pragma unroll
        for (int r = 0; r < R; ++r) lp[r] = -(s[r] + gconst);
    };
    if (want_lp && (A.flags & B2F_FLOW_LOGP_OF_INPUT)) base_logp(xin ? xin : x0, false);

    // ---- the layers ------------------------------------------------------------------------------------------------
    int run = 0, flip = 0;
    for (int oi = 0; oi < A.n_ops; ++oi) {
        const DevOp& op = A.ops[oi];
        if (op.kind == B2F_OP_FLIP) { flip ^= 1; continue; }
        if (op.kind == B2F_OP_ELEMENTWISE) {
            while (oi + 1 < A.n_ops && A.ops[oi + 1].kind == B2F_OP_ELEMENTWISE) ++oi;
            if (er) {                               // two runs separated only by FLIPs (no preset does this): apply the first
                for (int c0 = 0; c0 < D; c0 += 4) {
#pragma unroll
                    for (int r = 0; r < R; ++r) {
                        float xv[4];
                        ld4(x0 + r * 32 * XS, c0, xv);
                        apply_run(er, D, c0, xv);
                        st4(x0 + r * 32 * XS, c0, xv);
                    }
                }
            }
            er = ea + (size_t)run * 2 * D;
            ++run;
            continue;
        }
        rows_layer<MODE, HP, R, RQ>(wbuf + A.woff[oi], x0, XS, D, flip, op, er, ld, wst, A.rq_stride, xin, live);
        er = nullptr;
        xin = nullptr;                                   // later layers read what this one wrote
    }

    // ---- epilogue ------------------------------------------------------------------------------------------------
    if (inplace) {
        // the rows are already where they belong; the host guarantees an even number of flips and at least one layer
        if (want_lp && !(A.flags & B2F_FLOW_LOGP_OF_INPUT)) base_logp(x0, er != nullptr);
        else if (er) {
            for (int c0 = 0; c0 < D; c0 += 4) {
                float xv[4];
                if (live) { ld4(x0, c0, xv); apply_run(er, D, c0, xv); st4(x0, c0, xv); }
            }
        }
    } else if (want_lp && !(A.flags & B2F_FLOW_LOGP_OF_INPUT)) base_logp(x0, false);
#pragma unroll
    for (int r = 0; r < R; ++r) {
        const int m = r * 32 + lane;
        if (m < rows) {
            const float l = ld[r] + ldc;
            if (A.log_det) A.log_det[wrow0 + m] = l;
            if (want_lp) A.log_prob[wrow0 + m] = lp[r] + l;
        }
    }
    if (A.y && !inplace) {
        __syncwarp();
        float4* dst = reinterpret_cast<float4*>(A.y + wrow0 * D);
        int m = 0, c4 = lane;
        while (c4 >= D4) { c4 -= D4; ++m; }
        for (int idx = lane; m < rows; idx += 32) {
            // logical columns 4*c4 .. 4*c4+3 of the output row
            const int c0 = flip ? D - 4 - 4 * c4 : 4 * c4;
            float v[4];
            ld4(xw + m * XS, c0, v);
            if (er) apply_run(er, D, c0, v);
            __stcs(dst + idx, flip ? make_float4(v[3], v[2], v[1], v[0]) : make_float4(v[0], v[1], v[2], v[3]));
            c4 += 32;
            while (c4 >= D4) { c4 -= D4; ++m; }
        }
    }
  }   // tiles of this warp
}

template <int MODE, int HP4, bool RQ, int NT>
static cudaError_t launch_rows_kernel(const RowsArgs& A, unsigned grid, size_t smem, cudaStream_t st) {
    auto kern = flow_rows_kernel<MODE, HP4, 1, RQ, NT>;
    cudaError_t ce = (cudaError_t)raise_smem_limit((const void*)kern, smem);
    if (ce != cudaSuccess) return ce;
    kern<<<grid, NT, smem, st>>>(A);
    return cudaSuccess;
}

constexpr int kRowsThreadsAffine = 128, kRowsThreadsSpline = 64;
// one-pass affine / shift programs whose row tile, not the register file, limits the resident warps (MAF-128: 17 KB of tile per
// warp + 25 KB of weights = two 4-warp CTAs per SM): ONE 12-warp CTA shares the weights and fills the shared memory
constexpr int kRowsThreadsAffineBig = 384;

}  // namespace b2f
