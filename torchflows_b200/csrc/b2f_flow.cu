// Whole-flow fused kernel (generic FP32/FFMA path): one launch applies every layer of a
// BijectiveComposition to a tile of samples that stays in shared memory, and finishes with the base
// log-density.  Conditioner outputs (the transformer parameters h) only ever exist in registers.
//
// Replaces (file:line relative to /root/reference/torchflows):
//   bijections/base.py:203-232                 BijectiveComposition.forward / inverse (layer loop, log-det sum)
//   bijections/finite/autoregressive/layers_base.py:119-163   CouplingBijection (HalfSplit partition, clone, scatter)
//   .../layers_base.py:202-223                 MaskedAutoregressiveBijection one-pass and D-step sequential direction
//   .../layers_base.py:300-318, layers.py:19-69  ElementwiseAffine / ActNorm with broadcast global parameters
//   .../conditioning/transforms.py:197-198,259-264,293-307   MADE / FeedForward (Linear-Tanh-Linear)
//   bijections/finite/matrix/permutation.py:19-37   ReversePermutationMatrix (folded into column addressing)
//   flows.py:628-648, base_distributions/gaussian.py:46-54   log_prob = base log-density + log-det
//
// Data layout in HBM: x, y are (B, D) fp32 row-major; one CTA owns TM consecutive rows (one contiguous
// TM*D*4-byte block).  In shared memory the tile is [TM][XS] with XS = D|1 (odd stride: a warp that walks
// 32 samples of one column and a warp that walks 32 columns of one sample are both bank-conflict free).
// Thread mapping of the conditioner + transformer phase: a warp = 32 samples x one target element, so every
// weight address is warp-uniform (one broadcast 16-byte load feeds 4 FFMAs in 32 lanes); a thread owns a
// sample, so its log-det partial needs no cross-lane traffic; warps that share a sample group combine
// their partials through shared memory in a fixed order (deterministic).  The final per-row reduction of
// the Gaussian base density is a warp-shuffle (xor butterfly) reduction over columns.
#include <stdlib.h>
#include <string.h>

#include <algorithm>

#include "b2f_flow_device.cuh"

namespace b2f {

struct FlowArgs {
    DevOp ops[B2F_MAX_OPS];
    int n_ops, D, TM, logTM, XS, HS, WPG, G, has_seq, flags;
    long long B;
    const float* x;
    float* y;
    float* log_det;
    float* log_prob;
    const float* base_loc;
    const float* base_log_scale;
};

template <int MODE>
__device__ __forceinline__ void run_transform(const Tile& t, const DevOp& op, int t0, int n_tgt, bool seq) {
#define B2F_CASE(TKV)                                                   \
    case TKV:                                                           \
        if (seq) sequential_pass<TKV, MODE>(t, op);                     \
        else transform_pass<TKV, MODE>(t, op, t0, n_tgt);               \
        break;
    switch (op.tkind) {
        B2F_CASE(B2F_T_SHIFT_ADD)
        B2F_CASE(B2F_T_SHIFT_SUB)
        B2F_CASE(B2F_T_AFFINE_FWD)
        B2F_CASE(B2F_T_AFFINE_INV)
        B2F_CASE(B2F_T_RQ_FWD)
        B2F_CASE(B2F_T_RQ_INV)
        B2F_CASE(B2F_T_LRS_FWD)
        B2F_CASE(B2F_T_LRS_INV)
    }
#undef B2F_CASE
}

template <int MODE>
__global__ void __launch_bounds__(512) flow_kernel(const __grid_constant__ FlowArgs A) {
    extern __shared__ __align__(16) float smem[];
    Tile t;
    t.D = A.D; t.TM = A.TM; t.logTM = A.logTM; t.XS = A.XS; t.HS = A.HS; t.WPG = A.WPG; t.G = A.G; t.flip = 0;
    t.xt = smem;
    t.hid = t.xt + A.TM * A.XS;
    t.act = t.hid + A.TM * A.HS;
    t.ldp = t.act + (A.has_seq ? A.TM * A.HS : 0);
    float* ldacc = t.ldp + A.WPG * A.TM;   // [TM] per-sample log-det
    float* lpin = ldacc + A.TM;            // [TM] base log-density of the input rows (LOGP_OF_INPUT)
    float* ea = lpin + A.TM;               // [3*D] alpha / beta / log alpha of the current elementwise layer
    float* ldc = ea + 3 * A.D;             // [1]  batch-independent log-det of the elementwise layers

    const int tid = threadIdx.x, NT = blockDim.x, lane = tid & 31, warp = tid >> 5, NW = NT >> 5;
    const int D = A.D, TM = A.TM, XS = A.XS;
    const long long row0 = (long long)blockIdx.x * TM;
    const int rows = (int)min((long long)TM, A.B - row0);

    // ---- load the tile (coalesced: a warp reads one row segment), rows beyond B are zero-filled -------
    const float* xg = A.x + row0 * D;
    if ((D & 3) == 0 && ((reinterpret_cast<uintptr_t>(A.x) & 15) == 0)) {
        for (int m = warp; m < TM; m += NW) {
            float* dst = t.xt + m * XS;
            if (m < rows) {
                const float4* src = reinterpret_cast<const float4*>(xg + (size_t)m * D);
                for (int j4 = lane; j4 < (D >> 2); j4 += 32) {
                    const float4 v = __ldg(src + j4);
                    dst[4 * j4 + 0] = v.x; dst[4 * j4 + 1] = v.y; dst[4 * j4 + 2] = v.z; dst[4 * j4 + 3] = v.w;
                }
            } else {
                for (int j = lane; j < D; j += 32) dst[j] = 0.0f;
            }
        }
    } else {
        for (int m = warp; m < TM; m += NW) {
            float* dst = t.xt + m * XS;
            for (int j = lane; j < D; j += 32) dst[j] = (m < rows) ? __ldg(xg + (size_t)m * D + j) : 0.0f;
        }
    }
    if (tid < TM) ldacc[tid] = 0.0f;
    if (tid == 0) ldc[0] = 0.0f;
    __syncthreads();

    const bool want_lp = A.log_prob != nullptr;
    auto base_logp_rows = [&](float* dst) {
        // DiagonalGaussian.log_prob (gaussian.py:46-54): warp per row, lanes over columns, shuffle reduction
        for (int m = warp; m < TM; m += NW) {
            const float* xr = t.xt + m * XS;
            float s = 0.0f;
            for (int j = lane; j < D; j += 32) {
                const float loc = A.base_loc ? __ldg(A.base_loc + j) : 0.0f;
                const float lsc = A.base_log_scale ? __ldg(A.base_log_scale + j) : 0.0f;
                s += gauss_logp(xr[t.col(j)], loc, lsc);
            }
            s = warp_sum(s);
            if (lane == 0) dst[m] = s;
        }
    };
    if (want_lp && (A.flags & B2F_FLOW_LOGP_OF_INPUT)) base_logp_rows(lpin);

    // ---- the layers --------------------------------------------------------------------------------
    for (int oi = 0; oi < A.n_ops; ++oi) {
        const DevOp& op = A.ops[oi];
        if (op.kind == B2F_OP_FLIP) { t.flip ^= 1; continue; }
        if (op.kind == B2F_OP_ELEMENTWISE && (op.flags & B2F_FLAG_ROW_BIAS)) {
            // context-conditioned elementwise layer (layers_base.py:281-296): its parameters were predicted per row, (B, D, 2)
            const float* pr = op.p0 + (size_t)row0 * D * 2;
            const bool fwd = op.tkind == B2F_T_AFFINE_FWD;
            for (int m = warp; m < TM; m += NW) {
                float* xr = t.xt + m * XS;
                float sld = 0.0f;
                if (m < rows) {
                    for (int j = lane; j < D; j += 32) {
                        const float2 u = __ldg(reinterpret_cast<const float2*>(pr + ((size_t)m * D + j) * 2));
                        float a, la;
                        affine_scale<0>(u.x, a, la);
                        const int c = t.col(j);
                        xr[c] = fwd ? fmaf(a, xr[c], u.y) : (xr[c] - u.y) / a;
                        sld += fwd ? la : -la;
                    }
                }
                sld = warp_sum(sld);
                if (lane == 0) ldacc[m] += sld;
            }
            __syncthreads();
            continue;
        }
        if (op.kind == B2F_OP_ELEMENTWISE) {
            // (a per-row layer ends a run of global ones: it reports kind -1 to the run composer)
            auto get = [&](int i) { return EwOp{(A.ops[i].flags & B2F_FLAG_ROW_BIAS) ? -1 : A.ops[i].kind, A.ops[i].tkind, A.ops[i].p0}; };
            const int n_run = elementwise_stage_run(ea, get, oi, A.n_ops, D, tid, NT);
            __syncthreads();
            for (int m = warp; m < TM; m += NW) {
                float* xr = t.xt + m * XS;
                for (int j = lane; j < D; j += 32) {
                    const int c = t.col(j);
                    xr[c] = fmaf(ea[j], xr[c], ea[D + j]);
                }
            }
            if (warp == 0) {   // log-det of the run, identical for every sample
                float s = 0.0f;
                for (int j = lane; j < D; j += 32) s += ea[2 * D + j];
                s = warp_sum(s);
                if (lane == 0) ldc[0] += s;
            }
            __syncthreads();
            oi += n_run - 1;
            continue;
        }
        const bool coupling = op.kind == B2F_OP_COUPLING;
        const bool seq = op.kind == B2F_OP_MADE_SEQ;
        const int n_src = coupling ? D / 2 : D;            // HalfSplit: first D//2 flat dims are the source
        const int t0 = coupling ? D / 2 : 0, n_tgt = D - t0;
        if (!seq) {
            hidden_layer<true>(t, op, n_src, (op.flags & B2F_FLAG_ROW_BIAS) ? op.p1 + row0 * op.H : nullptr, rows);
            __syncthreads();
        }
        run_transform<MODE>(t, op, t0, n_tgt, seq);
        __syncthreads();
        if (tid < TM) {
            float s = 0.0f;
            const int ns = seq ? 1 : t.WPG;
            for (int sl = 0; sl < ns; ++sl) s += t.ldp[sl * TM + tid];
            ldacc[tid] += s;
        }
        __syncthreads();
    }

    // ---- epilogue: outputs ---------------------------------------------------------------------------
    if (want_lp && !(A.flags & B2F_FLOW_LOGP_OF_INPUT)) {
        base_logp_rows(lpin);
    }
    __syncthreads();
    if (tid < rows) {
        const float ld = ldacc[tid] + ldc[0];
        if (A.log_det) A.log_det[row0 + tid] = ld;
        if (want_lp) A.log_prob[row0 + tid] = lpin[tid] + ld;
    }
    if (A.y) {
        float* yg = A.y + row0 * D;
        if ((D & 3) == 0 && ((reinterpret_cast<uintptr_t>(A.y) & 15) == 0)) {
            for (int m = warp; m < rows; m += NW) {
                const float* src = t.xt + m * XS;
                float4* dst = reinterpret_cast<float4*>(yg + (size_t)m * D);
                for (int j4 = lane; j4 < (D >> 2); j4 += 32) {
                    float4 v;
                    v.x = src[t.col(4 * j4 + 0)]; v.y = src[t.col(4 * j4 + 1)];
                    v.z = src[t.col(4 * j4 + 2)]; v.w = src[t.col(4 * j4 + 3)];
                    dst[j4] = v;
                }
            }
        } else {
            for (int m = warp; m < rows; m += NW)
                for (int j = lane; j < D; j += 32) yg[(size_t)m * D + j] = t.xt[m * XS + t.col(j)];
        }
    }
}

static int ilog2(int v) { int l = 0; while ((1 << l) < v) ++l; return l; }

}  // namespace b2f

namespace b2f {
int try_launch_flow_tc(const b2f_op_t* ops, int32_t n_ops, const float* x, float* y, float* log_det, float* log_prob,
                       const float* base_loc, const float* base_log_scale, int64_t B, int32_t D, int32_t flags,
                       void* stream, float* ws);   // b2f_flow_tc.cu (ws: optional save area for the layer inputs)
int try_launch_flow_tcq(const b2f_op_t* ops, int32_t n_ops, const float* x, float* y, float* log_det, float* log_prob,
                        int64_t B, int32_t D, int32_t flags, void* stream, const TcqNoise* noise);   // b2f_flow_tcq.cu
int try_launch_flow_tca(const b2f_op_t* ops, int32_t n_ops, const float* x, float* y, float* log_det, float* log_prob,
                        int64_t B, int32_t D, int32_t flags, void* stream, const TcqNoise* noise);   // b2f_flow_tca.cu
int try_launch_flow_tcm(const b2f_op_t* ops, int32_t n_ops, const float* x, float* y, float* log_det, float* log_prob,
                        int64_t B, int32_t D, int32_t flags, void* stream, const TcqNoise* noise);   // b2f_flow_tcm.cu
int try_launch_flow_rows(const b2f_op_t* ops, int32_t n_ops, const float* x, float* y, float* log_det, float* log_prob,
                         const float* base_loc, const float* base_log_scale, int64_t B, int32_t D, int32_t flags,
                         void* stream);  // b2f_flow_rows.cu
}

using namespace b2f;

static int flow_apply_impl(const b2f_op_t* ops, int32_t n_ops, const float* x, float* y, float* log_det,
                           float* log_prob, const float* base_loc, const float* base_log_scale, int64_t B,
                           int32_t D, int32_t flags, void* stream, float* ws, int32_t* saved) {
    if (B == 0 && n_ops >= 0 && D > 0) return B2F_OK;      // empty batch: nothing to do (pointers may be null)
    if (!ops || n_ops < 0 || !x || D <= 0 || B < 0) return fail(B2F_ERR_INVALID, "b2f_flow_apply: bad arguments");
    if (n_ops > B2F_MAX_OPS) return fail(B2F_ERR_UNSUPPORTED, "b2f_flow_apply: %d ops > B2F_MAX_OPS", n_ops);
    if (B == 0) return B2F_OK;
    {
        // Spline programs (23 parameters per element: the output layer is a real GEMM) go to the tcgen05 kernel first,
        // affine / shift programs and anything with a sequential layer to the row-per-thread kernel first; what neither
        // takes runs on the generic kernel below.  Linear rational spline programs are not RQ programs here: every
        // tensor-core kernel declines them by transformer kind, the row-per-thread kernel takes their sequential inverse.
        bool has_rq = false;
        for (int i = 0; i < n_ops; ++i)
            if (ops[i].kind >= B2F_OP_COUPLING && (ops[i].tkind == B2F_T_RQ_FWD || ops[i].tkind == B2F_T_RQ_INV)) has_rq = true;
        if (has_rq && !ws) {       // programs laid out for the second-generation spline kernel (B2F_FLAG_TCQ_OPERANDS)
            const int rc = try_launch_flow_tcq(ops, n_ops, x, y, log_det, log_prob, B, D, flags, stream, nullptr);
            if (rc == 1) last_flow_kernel() = B2F_KERNEL_TCQ;
            if (rc != 0) return rc == 1 ? B2F_OK : rc;
            const int rm = try_launch_flow_tcm(ops, n_ops, x, y, log_det, log_prob, B, D, flags, stream, nullptr);
            if (rm == 1) last_flow_kernel() = B2F_KERNEL_TCM;
            if (rm != 0) return rm == 1 ? B2F_OK : rm;
        }
        if (!has_rq && !ws) {      // affine / shift coupling programs laid out for the multi-tile tensor-core kernel
            const int rc = try_launch_flow_tca(ops, n_ops, x, y, log_det, log_prob, B, D, flags, stream, nullptr);
            if (rc == 1) last_flow_kernel() = B2F_KERNEL_TCA;
            if (rc != 0) return rc == 1 ? B2F_OK : rc;
        }
        for (int attempt = 0; attempt < 2; ++attempt) {
            const bool tc = has_rq ? attempt == 0 : attempt == 1;
            const int rc = tc ? try_launch_flow_tc(ops, n_ops, x, y, log_det, log_prob, base_loc, base_log_scale, B, D, flags, stream, ws)
                              : try_launch_flow_rows(ops, n_ops, x, y, log_det, log_prob, base_loc, base_log_scale, B, D, flags, stream);
            if (rc == 1) last_flow_kernel() = tc ? B2F_KERNEL_TC : B2F_KERNEL_ROWS;
            if (rc == 1 && tc && ws && saved) *saved = 1;
            if (rc != 0) return rc == 1 ? B2F_OK : rc;
        }
    }
    for (int i = 0; i < n_ops; ++i)
        if (ops[i].flags & B2F_FLAG_SEQ_FOLDED)
            return fail(B2F_ERR_UNSUPPORTED, "b2f_flow_apply: op %d carries folded sequential-spline operands (B2F_FLAG_SEQ_FOLDED), "
                        "which only the row-per-thread kernel takes, and that kernel declined this program", i);
    FlowArgs A;
    memset(&A, 0, sizeof(A));
    int Hmax = 1, has_seq = 0, has_spline = 0;
    for (int i = 0; i < n_ops; ++i) {
        const b2f_op_t& o = ops[i];
        DevOp& d = A.ops[i];
        d.kind = o.kind; d.tkind = o.tkind; d.H = o.n_hidden; d.flags = o.flags; d.boundary = o.boundary;
        d.p0 = (const float*)o.p[0]; d.p1 = (const float*)o.p[1]; d.p2 = (const float*)o.p[2];
        d.p3 = (const float*)o.p[3]; d.p4 = (const int*)o.p[4];
        switch (o.kind) {
            case B2F_OP_FLIP: break;
            case B2F_OP_ELEMENTWISE:
                if (!o.p[0]) return fail(B2F_ERR_INVALID, "op %d: elementwise layer without parameters", i);
                if (o.tkind != B2F_T_AFFINE_FWD && o.tkind != B2F_T_AFFINE_INV)
                    return fail(B2F_ERR_UNSUPPORTED, "op %d: elementwise transformer kind %d", i, o.tkind);
                break;
            case B2F_OP_COUPLING: case B2F_OP_MADE: case B2F_OP_MADE_SEQ: {
                if (!o.p[0] || !o.p[1] || !o.p[2] || !o.p[3] || o.n_hidden <= 0)
                    return fail(B2F_ERR_INVALID, "op %d: conditioner parameters missing", i);
                if (params_per_element(o.tkind, 8) < 0) return fail(B2F_ERR_INVALID, "op %d: transformer kind", i);
                const bool rq = o.tkind == B2F_T_RQ_FWD || o.tkind == B2F_T_RQ_INV;
                const bool lrs = o.tkind == B2F_T_LRS_FWD || o.tkind == B2F_T_LRS_INV;
                if (o.tkind == B2F_T_SCALE_FWD || o.tkind == B2F_T_SCALE_INV)
                    return fail(B2F_ERR_UNSUPPORTED, "op %d: transformer kind %d has no flow-program kernel", i, o.tkind);
                if (rq && o.n_bins != 8)
                    return fail(B2F_ERR_UNSUPPORTED, "op %d: fused RQ spline needs n_bins == 8 (got %d)", i, o.n_bins);
                if (lrs && o.n_bins != 8)
                    return fail(B2F_ERR_UNSUPPORTED, "op %d: fused linear rational spline needs n_bins == 8 (got %d)", i, o.n_bins);
                if ((rq || lrs) && !(o.boundary > 0.0f)) return fail(B2F_ERR_INVALID, "op %d: boundary", i);
                if (o.kind == B2F_OP_COUPLING && D < 2) return fail(B2F_ERR_INVALID, "op %d: coupling needs D >= 2", i);
                if (o.kind == B2F_OP_MADE_SEQ) { if (!o.p[4]) return fail(B2F_ERR_INVALID, "op %d: finalisation steps", i); has_seq = 1; }
                if ((rq || lrs) && (reinterpret_cast<uintptr_t>(o.p[2]) & 15))
                    return fail(B2F_ERR_INVALID, "op %d: W2 tile layout must be 16-byte aligned", i);
                has_spline |= rq || lrs;
                Hmax = std::max(Hmax, o.n_hidden);
                break;
            }
            default: return fail(B2F_ERR_INVALID, "op %d: unknown kind %d", i, o.kind);
        }
    }
    A.n_ops = n_ops; A.D = D; A.B = B; A.flags = flags; A.has_seq = has_seq;
    A.x = x; A.y = y; A.log_det = log_det; A.log_prob = log_prob; A.base_loc = base_loc; A.base_log_scale = base_log_scale;
    A.XS = D | 1; A.HS = Hmax | 1;
    // tile shape: a sample group is one warp wide; WPG warps share a group and split its target elements
    int TM, NT;
    if (has_seq) { TM = 64; NT = 64; }          // sequential op: thread == sample, every warp busy
    else if (D <= 32) { TM = 128; NT = 256; }
    else { TM = 64; NT = has_spline ? 512 : 256; }
    if (const char* e = getenv("B2F_TM")) TM = atoi(e);
    if (const char* e = getenv("B2F_NT")) NT = atoi(e);
    auto smem_bytes = [&](int tm, int nt) {
        const int wpg = (nt / 32) / (tm / 32);
        return (size_t)sizeof(float) * ((size_t)tm * A.XS + (size_t)tm * A.HS * (has_seq ? 2 : 1) + (size_t)wpg * tm +
                                        2 * tm + 3 * D + 4);
    };
    while (TM > 32 && smem_bytes(TM, NT) > 200 * 1024) { TM >>= 1; if (NT > TM * 16) NT = TM * 16; }
    if (TM < 32 || (TM & (TM - 1)) || NT % 32 || NT > 512 || (NT / 32) % (TM / 32) || NT / 32 < TM / 32)
        return fail(B2F_ERR_INVALID, "b2f_flow_apply: bad tile shape TM=%d NT=%d", TM, NT);
    const size_t smem = smem_bytes(TM, NT);
    if (smem > 227 * 1024) return fail(B2F_ERR_UNSUPPORTED, "b2f_flow_apply: D=%d H=%d does not fit shared memory", D, Hmax);
    A.TM = TM; A.logTM = ilog2(TM); A.G = TM / 32; A.WPG = (NT / 32) / A.G;
    const long long grid = (B + TM - 1) / TM;
    if (grid > 0x7fffffffLL) return fail(B2F_ERR_UNSUPPORTED, "b2f_flow_apply: batch too large for one launch");
    auto kern = (flags & B2F_FLOW_MODE_PRECISE) ? flow_kernel<0> : ((flags & B2F_FLOW_MODE_FAST_KNOTS) ? flow_kernel<2> : flow_kernel<1>);
    cudaError_t ce = (cudaError_t)raise_smem_limit((const void*)kern, smem);
    if (ce != cudaSuccess) return fail(B2F_ERR_CUDA, "cudaFuncSetAttribute: %s", cudaGetErrorString(ce));
    kern<<<(unsigned)grid, NT, smem, (cudaStream_t)stream>>>(A);
    last_flow_kernel() = B2F_KERNEL_GENERIC;
    return check_launch("b2f_flow_apply");
}

extern "C" int b2f_flow_apply(const b2f_op_t* ops, int32_t n_ops, const float* x, float* y, float* log_det,
                              float* log_prob, const float* base_loc, const float* base_log_scale, int64_t B,
                              int32_t D, int32_t flags, void* stream) {
    return flow_apply_impl(ops, n_ops, x, y, log_det, log_prob, base_loc, base_log_scale, B, D, flags, stream, nullptr, nullptr);
}

extern "C" int b2f_flow_apply_saving(const b2f_op_t* ops, int32_t n_ops, const float* x, float* y, float* log_det,
                                     float* log_prob, const float* base_loc, const float* base_log_scale, void* workspace,
                                     int32_t* saved, int64_t B, int32_t D, int32_t flags, void* stream) {
    if (!saved) return fail(B2F_ERR_INVALID, "b2f_flow_apply_saving: saved is null");
    *saved = 0;
    return flow_apply_impl(ops, n_ops, x, y, log_det, log_prob, base_loc, base_log_scale, B, D, flags, stream,
                           (float*)workspace, saved);
}

extern "C" int b2f_philox_normal(float* out, int64_t n_rows, int32_t D, const float* loc, const float* log_scale, uint64_t seed,
                                 uint64_t offset, void* stream);

extern "C" int b2f_flow_sample(const b2f_op_t* ops, int32_t n_ops, float* y, float* log_det, float* log_prob, const float* base_loc,
                               const float* base_log_scale, float* noise_scratch, int64_t B, int32_t D, int32_t flags,
                               uint64_t seed, uint64_t offset, void* stream) {
    if (B == 0 && n_ops >= 0 && D > 0) return B2F_OK;
    if (!ops || n_ops < 0 || D <= 0 || B < 0) return fail(B2F_ERR_INVALID, "b2f_flow_sample: bad arguments");
    if (n_ops > B2F_MAX_OPS) return fail(B2F_ERR_UNSUPPORTED, "b2f_flow_sample: %d ops > B2F_MAX_OPS", n_ops);
    if (D % 4 != 0 && !noise_scratch) return fail(B2F_ERR_UNSUPPORTED, "b2f_flow_sample: this shape needs a noise scratch buffer");
    // programs of the spline tensor-core kernel draw their tiles in registers: the noise never exists in memory
    TcqNoise nz;
    nz.seed = seed; nz.offset = offset; nz.base_loc = base_loc; nz.base_log_scale = base_log_scale;
    int rc = try_launch_flow_tcq(ops, n_ops, nullptr, y, log_det, log_prob, B, D, flags, stream, &nz);
    if (rc == 1) { last_flow_kernel() = B2F_KERNEL_TCQ; return B2F_OK; }
    if (rc != 0) return rc;
    rc = try_launch_flow_tca(ops, n_ops, nullptr, y, log_det, log_prob, B, D, flags, stream, &nz);
    if (rc == 1) { last_flow_kernel() = B2F_KERNEL_TCA; return B2F_OK; }
    if (rc != 0) return rc;
    rc = try_launch_flow_tcm(ops, n_ops, nullptr, y, log_det, log_prob, B, D, flags, stream, &nz);
    if (rc == 1) { last_flow_kernel() = B2F_KERNEL_TCM; return B2F_OK; }
    if (rc != 0) return rc;
    // every other program: the same stream, materialised once, then the ordinary launch
    if (!noise_scratch) return fail(B2F_ERR_UNSUPPORTED, "b2f_flow_sample: this program needs a noise scratch buffer of B * D floats");
    if ((rc = b2f_philox_normal(noise_scratch, B, D, base_loc, base_log_scale, seed, offset, stream)) != B2F_OK) return rc;
    return flow_apply_impl(ops, n_ops, noise_scratch, y, log_det, log_prob, base_loc, base_log_scale, B, D, flags, stream, nullptr, nullptr);
}
