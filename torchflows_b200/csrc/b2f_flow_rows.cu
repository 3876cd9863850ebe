// Row-per-thread whole-flow kernel: eligibility, shared-memory budget and launch (device code: b2f_flow_rows.cuh).
#include <stdlib.h>
#include <string.h>

#include <algorithm>

#include "b2f_flow_rows.cuh"

namespace b2f {

// b2f_flow_rows_rq.cu: the instantiations with sequential spline layers (mode 0 / 1 / 2, hidden width <= 15)
cudaError_t launch_rows_spline(int mode, int hp4, const RowsArgs& A, unsigned grid, size_t smem, cudaStream_t st);

template <int MODE, int NT>
static cudaError_t launch_rows_h(const RowsArgs& A, int hp4, unsigned grid, size_t smem, cudaStream_t st) {
    switch (hp4) {
        case 1: return launch_rows_kernel<MODE, 1, false, NT>(A, grid, smem, st);
        case 2: return launch_rows_kernel<MODE, 2, false, NT>(A, grid, smem, st);
        case 3: return launch_rows_kernel<MODE, 3, false, NT>(A, grid, smem, st);
        case 4: return launch_rows_kernel<MODE, 4, false, NT>(A, grid, smem, st);
        case 5: return launch_rows_kernel<MODE, 5, false, NT>(A, grid, smem, st);
        case 6: return launch_rows_kernel<MODE, 6, false, NT>(A, grid, smem, st);
        case 7: return launch_rows_kernel<MODE, 7, false, NT>(A, grid, smem, st);
        default: return launch_rows_kernel<MODE, 8, false, NT>(A, grid, smem, st);
    }
}

// Returns 0 = not eligible (caller falls through), 1 = launched, negative = error.
int try_launch_flow_rows(const b2f_op_t* ops, int32_t n_ops, const float* x, float* y, float* log_det, float* log_prob,
                         const float* base_loc, const float* base_log_scale, int64_t B, int32_t D, int32_t flags,
                         void* stream) {
    if (getenv("B2F_DISABLE_ROWS")) return 0;
    if (D % 8 != 0 || D > 1024) return 0;
    if ((reinterpret_cast<uintptr_t>(x) & 15) || (y && (reinterpret_cast<uintptr_t>(y) & 15))) return 0;
    RowsArgs A;
    memset(&A, 0, sizeof(A));
    int Hmax = 0, Hrq = 0, n_runs = 0, n_cond = 0, wst_floats = 0;
    bool prev_ew = false;
    for (int i = 0; i < n_ops; ++i) {
        const b2f_op_t& o = ops[i];
        DevOp& d = A.ops[i];
        d.kind = o.kind; d.tkind = o.tkind; d.H = o.n_hidden; d.flags = o.flags; d.boundary = o.boundary;
        d.p0 = (const float*)o.p[0]; d.p1 = (const float*)o.p[1]; d.p2 = (const float*)o.p[2];
        d.p3 = (const float*)o.p[3]; d.p4 = (const int*)o.p[4];
        const bool ew = o.kind == B2F_OP_ELEMENTWISE;
        if (ew && !prev_ew) ++n_runs;
        prev_ew = ew;
        switch (o.kind) {
            case B2F_OP_FLIP: break;
            case B2F_OP_ELEMENTWISE:
                if (!o.p[0] || (o.tkind != B2F_T_AFFINE_FWD && o.tkind != B2F_T_AFFINE_INV) || (o.flags & B2F_FLAG_ROW_BIAS)) return 0;
                break;
            case B2F_OP_COUPLING: case B2F_OP_MADE: case B2F_OP_MADE_SEQ: {
                if (!o.p[0] || !o.p[1] || !o.p[2] || !o.p[3] || o.n_hidden <= 0 || o.n_hidden > 32) return 0;
                if (o.flags & B2F_FLAG_ROW_BIAS) return 0;      // context-conditioned layers: generic kernel
                if (o.kind == B2F_OP_MADE_SEQ && !o.p[4]) return 0;
                if (o.tkind == B2F_T_RQ_FWD || o.tkind == B2F_T_RQ_INV || o.tkind == B2F_T_LRS_INV) {
                    // splines: only the D-step sequential direction (the one-pass direction has a real GEMM as its output
                    // layer and belongs on the tensor cores, or for the linear rational spline on the generic kernel)
                    if (o.kind != B2F_OP_MADE_SEQ || o.n_bins != 8 || !(o.boundary > 0.0f) || o.n_hidden > 15) return 0;
                    if (reinterpret_cast<uintptr_t>(o.p[2]) & 15) return 0;
                    if (o.tkind == B2F_T_LRS_INV && (o.flags & B2F_FLAG_SEQ_FOLDED)) return 0;    // no folded variant
                    Hrq = std::max(Hrq, o.n_hidden);
                    wst_floats = std::max(wst_floats, o.n_hidden * padded_params(params_per_element(o.tkind, 8)) +
                                                          padded_params(params_per_element(o.tkind, 8)));
                } else if (o.tkind != B2F_T_SHIFT_ADD && o.tkind != B2F_T_SHIFT_SUB && o.tkind != B2F_T_AFFINE_FWD &&
                           o.tkind != B2F_T_AFFINE_INV) {
                    return 0;
                }
                Hmax = std::max(Hmax, o.n_hidden);
                ++n_cond;
                break;
            }
            default: return 0;
        }
    }
    if (n_cond == 0) return 0;     // purely elementwise programs: the generic kernel is already bandwidth-bound
    const int hp4 = (Hmax + 1 + 3) / 4, HP = 4 * hp4;      // + 1: hidden slot H carries the output bias
    if (hp4 > 8) return 0;
    int XS = D + 4;
    if (((XS >> 2) & 1) == 0) XS += 4;     // XS/4 odd: conflict-free 16-byte row accesses across a warp
    const bool spline = Hrq > 0;
    if (spline && (hp4 > 4 || (flags & B2F_FLOW_MODE_PRECISE))) return 0;      // precise splines: generic kernel
    int NT = spline ? kRowsThreadsSpline : kRowsThreadsAffine;
    // staged weights of every conditioner layer: w1 [n_src][HP] + b1 [HP] + w2 [n_tgt*P][HP] (no w2 for spline layers)
    size_t wtotal = 0;
    for (int i = 0; i < n_ops; ++i) {
        const b2f_op_t& o = ops[i];
        if (o.kind != B2F_OP_COUPLING && o.kind != B2F_OP_MADE && o.kind != B2F_OP_MADE_SEQ) continue;
        const int n_src = o.kind == B2F_OP_COUPLING ? D / 2 : D, n_tgt = o.kind == B2F_OP_COUPLING ? D - D / 2 : D;
        const bool rq = o.tkind == B2F_T_RQ_FWD || o.tkind == B2F_T_RQ_INV || o.tkind == B2F_T_LRS_INV;
        const int P = (o.tkind == B2F_T_SHIFT_ADD || o.tkind == B2F_T_SHIFT_SUB) ? 1 : 2;
        A.woff[i] = (int)wtotal;
        wtotal += (size_t)n_src * HP + HP + (rq ? 0 : (size_t)n_tgt * P * HP);
    }
    const int R = 1;
    // Programs whose conditioner layers are ALL sequential (MAF / MA-RQNSF sampling) and that produce an output: the rows
    // live in the output buffer itself -- every thread walks its own row of y in global memory (L1 keeps its current
    // line) -- so no shared-memory tile limits the number of resident warps.  Needs: an even number of flips (the result
    // is already in logical order), every elementwise run followed by a layer or trailing, x and y distinct.
    bool inplace = y != nullptr && (const void*)y != (const void*)x && !getenv("B2F_ROWS_NO_INPLACE");
    if (inplace) {
        int nflip = 0, state = 0;      // state 0: no run pending, 1: run pending, 2: run pending and a flip seen after it
        for (int i = 0; i < n_ops && inplace; ++i) {
            const b2f_op_t& o = ops[i];
            if (o.kind == B2F_OP_FLIP) { ++nflip; if (state == 1) state = 2; continue; }
            if (o.kind == B2F_OP_ELEMENTWISE) { if (state == 2) inplace = false; state = 1; continue; }
            if (o.kind != B2F_OP_MADE_SEQ) inplace = false;   // one-pass layers walk a row twice: measured slower in place
            state = 0;
        }
        if (nflip & 1) inplace = false;
    }
    if (inplace && !spline) {
        // affine / shift programs: worth it only when the tile, not the register file, limits the resident warps
        const size_t with_tile = sizeof(float) * ((size_t)(NT / 32) * 32 * XS + (size_t)n_runs * 2 * D + 2 * D + 8 + wtotal);
        const size_t ctas = (220 * 1024) / with_tile;
        if (ctas * (NT / 32) >= 16) inplace = false;
    }
    if (inplace) XS = 0;                                           // no tile
    const int rq_stride = spline ? ((wst_floats + 3) & ~3) : 0;     // one element's output-layer block: H * PP + PP floats
    auto smem_for = [&](int nt) {
        return sizeof(float) * ((size_t)(nt / 32) * 32 * R * XS + (size_t)n_runs * 2 * D + 2 * D + std::max(8, 2 * (nt / 32)) +
                                wtotal + (size_t)(nt / 32) * 2 * rq_stride);        // (+ [2][warps] partials, >= 8 floats)
    };
    if (!spline && !inplace && !getenv("B2F_ROWS_NO_BIG_CTA")) {
        // tile-limited programs: one big CTA per SM holds more warps than several small ones that each stage the weights
        const size_t small = smem_for(NT), big = smem_for(kRowsThreadsAffineBig);
        const size_t warps_small = small <= 110 * 1024 ? std::min<size_t>((227 * 1024) / small, 16) * (NT / 32) : 0;
        if (big <= 227 * 1024 && (size_t)(kRowsThreadsAffineBig / 32) > warps_small) NT = kRowsThreadsAffineBig;
    }
    const size_t smem = smem_for(NT);
    if (smem > (NT == kRowsThreadsAffineBig ? 227 : 110) * 1024) return 0;
    A.n_ops = n_ops; A.D = D; A.XS = XS; A.B = B; A.flags = flags; A.n_runs = n_runs;
    A.wtotal = (int)wtotal; A.rq_stride = rq_stride; A.inplace = inplace ? 1 : 0;
    A.x = x; A.y = y; A.log_det = log_det; A.log_prob = log_prob; A.base_loc = base_loc; A.base_log_scale = base_log_scale;
    // a warp walks tiles_per_warp consecutive 32-row tiles (the per-CTA weight staging is amortised over them) while the
    // grid stays several waves deep, so that the hardware CTA scheduler still balances the SMs
    int sms = 148;
    { int dev = 0; if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev); }
    const long long warp_tiles = (B + 32 * R - 1) / (32 * R);
    long long tpw = warp_tiles / ((long long)sms * 16 * 3);          // ~16 resident warps per SM, >= 3 waves
    tpw = std::max(1LL, std::min(8LL, tpw));
    if (const char* e = getenv("B2F_ROWS_TPW")) { const int t = atoi(e); if (t >= 1 && t <= 64) tpw = t; }
    A.tiles_per_warp = (int)tpw;
    const long long rows_per_cta = (long long)(NT / 32) * 32 * R * tpw;
    const long long grid = (B + rows_per_cta - 1) / rows_per_cta;
    if (grid > 0x7fffffffLL) return fail(B2F_ERR_UNSUPPORTED, "b2f_flow_apply: batch too large for one launch");
    cudaStream_t st = (cudaStream_t)stream;
    const int mode = (flags & B2F_FLOW_MODE_PRECISE) ? 0 : ((flags & B2F_FLOW_MODE_FAST_KNOTS) ? 2 : 1);
    const cudaError_t ce = spline ? launch_rows_spline(mode, hp4, A, (unsigned)grid, smem, st)
                         : NT == kRowsThreadsAffineBig
                             ? (mode == 0 ? launch_rows_h<0, kRowsThreadsAffineBig>(A, hp4, (unsigned)grid, smem, st)
                                          : launch_rows_h<1, kRowsThreadsAffineBig>(A, hp4, (unsigned)grid, smem, st))
                             : (mode == 0 ? launch_rows_h<0, kRowsThreadsAffine>(A, hp4, (unsigned)grid, smem, st)
                                          : launch_rows_h<1, kRowsThreadsAffine>(A, hp4, (unsigned)grid, smem, st));
    if (ce != cudaSuccess) return fail(B2F_ERR_CUDA, "flow_rows_kernel: %s", cudaGetErrorString(ce));
    const int rc = check_launch("b2f_flow_apply (rows kernel)");
    return rc == B2F_OK ? 1 : rc;
}

}  // namespace b2f
