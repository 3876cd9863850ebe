/* b2f.h -- C ABI of libb2f.so: hand-written sm_100a kernels for the coupling / masked-autoregressive
 * bijection hot path of torchflows (v1.2.0), called from torchflows_b200's torch.autograd.Functions.
 *
 * The reference has no FFI boundary (it is pure Python on PyTorch eager); the entry points below are
 * what a maintainer would bind with ctypes from the reference's own classes (see INTEGRATION.md).
 * Each one names the reference code it replaces, file:line relative to /root/reference/torchflows.
 *
 * Conventions (all entry points):
 *   - plain pointers to DEVICE memory (fp32, contiguous, row-major), sizes as integers, `stream` is a
 *     cudaStream_t passed as void*; no torch types;
 *   - the caller owns every buffer; kernels read inputs, write outputs; no allocation, no host sync;
 *   - return 0 on success, a negative B2F_ERR_* code otherwise; b2f_last_error() gives the message of
 *     the last failure on the calling thread;  nothing throws;
 *   - there is no CPU path: without a CUDA device every compute entry point fails with B2F_ERR_CUDA.
 */
#ifndef B2F_H_
#define B2F_H_
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B2F_OK 0
#define B2F_ERR_INVALID (-1)     /* bad shape / null pointer / inconsistent arguments */
#define B2F_ERR_UNSUPPORTED (-2) /* configuration outside the fused hot path */
#define B2F_ERR_CUDA (-3)        /* CUDA runtime error (message in b2f_last_error) */

/* Formula applied to each transformed element (transformers/linear/affine.py, transformers/spline/). */
enum b2f_transformer {
    B2F_T_SHIFT_ADD = 0,  /* Shift.forward           z = x + u0              affine.py:149-153 */
    B2F_T_SHIFT_SUB = 1,  /* Shift.inverse           x = z - u0              affine.py:155-159 */
    B2F_T_AFFINE_FWD = 2, /* Affine.forward / InverseAffine.inverse  z = a*x + u1, ld = +log a   affine.py:39-48 */
    B2F_T_AFFINE_INV = 3, /* Affine.inverse / InverseAffine.forward  x = (z-u1)/a, ld = -log a   affine.py:50-59 */
    B2F_T_RQ_FWD = 4,     /* RationalQuadratic.forward   spline/base.py:53-60, rational_quadratic.py:65-128 */
    B2F_T_RQ_INV = 5,     /* RationalQuadratic.inverse   spline/base.py:65-72, rational_quadratic.py:130-200 */
    B2F_T_LRS_FWD = 6,    /* LinearRational.forward      spline/linear_rational.py:92-135; 4 * n_bins parameters per element */
    B2F_T_LRS_INV = 7,    /* LinearRational.inverse      spline/linear_rational.py:137-182 */
    /* stand-alone transformer entry points only (b2f_transformer_apply / _backward), not flow programs: */
    B2F_T_SCALE_FWD = 8,  /* Scale.forward               z = a*x, ld = +log a    affine.py:186-193 */
    B2F_T_SCALE_INV = 9   /* Scale.inverse               x = z/a, ld = -log a    affine.py:195-202 */
};

/* One step of a flow program = one layer of BijectiveComposition (bijections/base.py:203-232) applied
 * in the direction the caller chose. */
enum b2f_op_kind {
    B2F_OP_ELEMENTWISE = 0, /* ElementwiseAffine / ActNorm with global parameters  layers_base.py:300-318, layers.py:19-69
                               p[0] = value (D,2); tkind = AFFINE_FWD or AFFINE_INV */
    B2F_OP_FLIP = 1,        /* ReversePermutationMatrix forward or inverse         matrix/permutation.py:19-37 */
    B2F_OP_COUPLING = 2,    /* CouplingBijection with HalfSplit + FeedForward(n_layers=2, Tanh)
                               layers_base.py:119-163, coupling_masks.py:78-81, transforms.py:293-307
                               p[0]=W1 (H,Ds)  p[1]=b1 (H)  p[2]=W2 tile layout (Dt,H,PP)  p[3]=b2 (Dt*P) */
    B2F_OP_MADE = 3,        /* MaskedAutoregressiveBijection, one-pass direction    layers_base.py:202-211, transforms.py:184-266
                               p[0]=W1*mask (H,D)  p[1]=b1  p[2]=(W2*mask) tile layout (D,H,PP)  p[3]=b2 (D*P) */
    B2F_OP_MADE_SEQ = 4     /* the D-step sequential direction                      layers_base.py:213-223
                               as B2F_OP_MADE plus p[4] = int32 finalisation step of each hidden unit (H) */
};

/* (op kind, tkind, n_bins) combinations that flow programs accept (b2f_flow_apply, b2f_flow_sample, b2f_flow_apply_saving,
 * b2f_flow_backward):
 *   ELEMENTWISE           AFFINE_FWD / AFFINE_INV                                   n_bins ignored
 *   COUPLING, MADE        SHIFT_*, AFFINE_*                                         n_bins ignored
 *   COUPLING, MADE        RQ_FWD / RQ_INV, LRS_FWD / LRS_INV                        n_bins == 8, boundary > 0
 *   MADE_SEQ              SHIFT_*, AFFINE_*                                         n_bins ignored
 *   MADE_SEQ              RQ_FWD / RQ_INV, LRS_FWD / LRS_INV                        n_bins == 8, boundary > 0
 *                         (b2f_flow_backward: RQ_INV / LRS_INV only, with B2F_FLAG_SEQ_LOGDET_EXACT)
 * SCALE_* are stand-alone transformer kinds only.  Linear rational spline (LRS) programs run on the generic FP32 kernel
 * (B2F_KERNEL_GENERIC); a MADE_SEQ LRS_INV layer with n_hidden <= 15 runs on the row-per-thread kernel (B2F_KERNEL_ROWS).
 * The tensor-core kernels decline LRS ops. */

/* W2 "tile layout": the reference's last Linear weight (Dt*P, H) (output index e*P+p, layers_base.py:143)
 * re-laid-out as [e][j][p] with p padded to PP = b2f_padded_params(P), so that the P parameters of one
 * element for one hidden unit are one aligned vector. */

#define B2F_MAX_OPS 40
#define B2F_FLAG_SEQ_LOGDET_EXACT 1 /* op flag: MADE_SEQ sums the true per-dimension log-dets instead of
                                       reproducing the reference's last-iteration value (SURVEY App. B.3) */

#define B2F_FLAG_TC_OPERANDS 2      /* op flag (COUPLING, RQ): p[4], p[5] hold the tensor-core operand layouts:
                                       p[4] = W1c: UMMA canonical K-major [32 x D/2] fp32 rounded to tf32 (rows >= H zero;
                                              column k = physical index inside the source half);
                                       p[5] = W2c: D/2/8 chunks, each canonical [192 x K2], K2 = roundup(H+2, 8):
                                              row = 24*(element in chunk) + parameter, columns 0..H-1 = W2, column H / H+1
                                              = tf32 hi / lo parts of b2, rest zero.  Byte offset of (row, k) in an operand
                                              with K columns: (row/8)*K*32 + (k/4)*128 + (row%8)*16 + (k%4)*4 */
#define B2F_FLAG_TC_FLIPPED 4       /* op flag: p[4] was laid out for a flipped tile (odd number of FLIP ops before) */
#define B2F_FLAG_TCQ_OPERANDS 8     /* op flag (COUPLING, RQ, n_bins 8), set on EVERY coupling op of a program made of
                                       ELEMENTWISE / FLIP / COUPLING ops: the program is laid out for the second-generation
                                       spline kernel (csrc/b2f_flow_tcq.cu; layout produced by torchflows_b200/_tcq.py):
                                       p[4] = layer blob (fp32 words, 16-byte aligned), with Dh = D/2, K2 = roundup(H+2, 8):
                                         [0,8)  int32 header: magic 'BTCQ', physical source half (0|1), 1 if the source half must be
                                                materialised (src affine below), H, K2, Dh/2 chunks, Dh, 0
                                         W1c    canonical [32 x Dh] tf32, columns in PHYSICAL order of the source half
                                         b1     32 floats (zero padded)
                                         W2c    Dh/2 chunks, each canonical [48 x K2]: row = 24*(element in chunk) + folded column
                                                (csrc/b2f_rqfast.cuh: log2e*u_x | log2e/1000*u_y | differences of padded derivative
                                                logits), elements in PHYSICAL order of the target half; K columns H, H+1 = bias hi, lo
                                         tgt    [Dh][8]: pre_a, pre_b (pending elementwise layers, applied when the element is read),
                                                post_a, post_b (elementwise layers that follow, applied at write-back), fin_a, fin_b
                                                (maps the written value to the standardised base-density argument; 0 unless this
                                                layer is the last writer of the column), 0, 0
                                         src    [Dh][2]: a, b of the pending elementwise layers on the source half
                                         misc   [4]: sup |log2e*u_x|, sup |log2e*u_y/1000|, sup |u_d/1000| over all inputs (from the weights;
                                                      the last includes the padded edge logit c/1000, 0 = no bound), 0
                                       p[5] (first coupling op) = program blob: int32 {magic, final pass on half 0, on half 1, layers},
                                         {sum of elementwise log-dets, base-density constant, 0, 0}, [D][2] final affine per physical
                                         column, [D][2] (exp(-log_scale), -loc*exp(-log_scale)) of the base density per column */

#define B2F_FLAG_TCA_OPERANDS 16    /* op flag (COUPLING, affine or shift), set on EVERY coupling op of a program made of
                                       ELEMENTWISE / FLIP / COUPLING ops: the program is laid out for the multi-tile affine kernel
                                       (csrc/b2f_flow_tca.cu; layout produced by torchflows_b200/_tca.py):
                                       p[4] = layer blob (fp32 words, 16-byte aligned), Dh = D/2, N1 = roundup(H, 16),
                                              K2 = roundup(H + 1, 8), N2 = roundup(Dh * P, 16), P = 2 (affine) or 1 (shift):
                                         [0,8)  int32 header: magic 'BTCA', physical source half, 1 if the source half must be
                                                materialised, H, N1, K2, Dh, P | inverse << 8
                                         W1hi, W1lo  canonical [N1 x Dh] each: tf32 hi / lo parts, columns in PHYSICAL order
                                         b1     32 floats (zero padded)
                                         W2hi, W2lo  canonical [N2 x K2] each: row = element * P + parameter (elements in PHYSICAL
                                                order of the target half), K column H = the bias
                                         tgt    [Dh][8] and src [Dh][2] as for B2F_FLAG_TCQ_OPERANDS
                                       p[5] (first coupling op) = program blob, as for B2F_FLAG_TCQ_OPERANDS */

#define B2F_FLAG_TCM_OPERANDS 32    /* op flag (MADE, RQ, n_bins 8, one-pass direction), set on EVERY MADE op of a program made of
                                       ELEMENTWISE / FLIP / MADE ops: the program is laid out for the masked-autoregressive spline
                                       kernel (csrc/b2f_flow_tcm.cu; layout produced by torchflows_b200/_tcm.py):
                                       p[4] = layer blob (fp32 words, 16-byte aligned), K2 = roundup(H+2, 8):
                                         [0,8)  int32 header: magic 'BTCM', 0, 1 if the tile must be materialised first (src affine
                                                below), H, K2, D/2 chunks, D, 0
                                         W1c    canonical [32 x D] tf32 of W1 * mask1, columns in PHYSICAL order
                                         b1     32 floats (zero padded)
                                         W2c    D/2 chunks, each canonical [48 x K2]: folded columns of (W2 * mask2, b2) as for
                                                B2F_FLAG_TCQ_OPERANDS, elements in PHYSICAL order
                                         tgt    [D][8], src [D][2], misc [4] as for B2F_FLAG_TCQ_OPERANDS
                                       p[5] (first MADE op) = program blob: int32 {magic, final pass, 0, layers}, then as for
                                         B2F_FLAG_TCQ_OPERANDS */

#define B2F_FLAG_ROW_BIAS 64        /* op flag (COUPLING): the conditioner is context-conditioned (conditioning/context.py:46-60,
                                       Concatenation: the hidden layer sees [x_A, context]).  p[0] holds the x_A columns of W1
                                       only, and p[1] is a PER-ROW hidden bias (B, H) = b1 + context . W1[:, n_src:]^T computed by
                                       the caller; b2f_flow_backward writes dL/d(pre-activation) per row into g[1] (B, H), from
                                       which the caller derives the gradients of b1, the context columns of W1 and the context.
                                       On an ELEMENTWISE op (context-conditioned ElementwiseAffine, layers_base.py:281-296): p[0]
                                       holds PER-ROW parameters (B, D, 2) predicted by the caller's conditioner, and the backward
                                       writes their gradient per row into g[0] (B, D, 2).
                                       Such programs run on the generic and backward kernels (b2f_flow.cu, b2f_flow_bwd.cu). */

#define B2F_FLAG_SEQ_FOLDED 128     /* op flag (MADE_SEQ, RQ, n_bins 8; inference): p[2] = folded output layer [element][hidden][24]
                                       (the 24 columns of csrc/b2f_rqfast.cuh, masks multiplied in, elements in LOGICAL order),
                                       p[3] = folded bias [element][24]; the sequential direction then evaluates the spline in the
                                       folded formulation of the tensor-core kernels (tolerance-checked like them) */

typedef struct b2f_op {
    int32_t kind;     /* enum b2f_op_kind */
    int32_t tkind;    /* enum b2f_transformer */
    int32_t n_hidden; /* H */
    int32_t n_bins;   /* RQ / LRS only (flow programs support 8; b2f_transformer_apply supports 1..64) */
    float boundary;   /* RQ / LRS only */
    int32_t flags;
    const void *p[6]; /* parameters, see enum b2f_op_kind */
    void *g[6];       /* b2f_flow_backward only: gradient buffers with the layout of p[i] (accumulated into) */
} b2f_op_t;

/* flags of b2f_flow_apply */
#define B2F_FLOW_LOGP_OF_INPUT 1 /* log_prob = base_log_prob(x_in) + log_det  (Flow.sample(return_log_prob=True),
                                    flows.py:710-712) instead of base_log_prob(y) + log_det (flows.py:646-648) */
#define B2F_FLOW_MODE_PRECISE 2  /* accurate libm-grade exp/log everywhere (default: SFU approximations after
                                    the bin search; knots and bin indices are identical in both modes) */

#define B2F_FLOW_MODE_FAST_KNOTS 4 /* opt-in: spline knots from SFU exponentials (ex2.approx) instead of the
                                     deterministic polynomial; ~25 %% fewer instructions per element, values within
                                     the same tolerances, but bin indices are no longer bit-reproducible on a CPU */

/* Runs `n_ops` layers over x:(B,D) in ONE kernel: y:(B,D) (nullable), log_det:(B) (nullable),
 * log_prob:(B) (nullable; adds the DiagonalGaussian log-density with base_loc / base_log_scale:(D),
 * both nullable = standard normal).  Replaces BijectiveComposition.forward / inverse
 * (bijections/base.py:203-232) + Flow.forward_with_log_prob (flows.py:628-648) + DiagonalGaussian.log_prob
 * (base_distributions/gaussian.py:46-54).  The caller lists ops in application order (for the inverse
 * direction: reversed layers with inverse transformer kinds). */
int b2f_flow_apply(const b2f_op_t *ops, int32_t n_ops, const float *x, float *y, float *log_det, float *log_prob,
                   const float *base_loc, const float *base_log_scale, int64_t B, int32_t D, int32_t flags,
                   void *stream);

/* Flow.sample with the base draws made by the library (flows.py:660-713, base_distributions/gaussian.py:41-44): the
 * program `ops` (inverse direction) is applied to z = base_loc + exp(base_log_scale) * n, n = standard normals from a
 * counter-based Philox4x32-10 stream (csrc/b2f_philox.cuh): flat element row * D + column is lane e % 4 of counter
 * e / 4 + offset under the 64-bit key `seed`.  Programs of the spline tensor-core kernel (B2F_KERNEL_TCQ) draw their
 * tiles in registers -- the noise is never written to or read from memory, a sample costs 4 D bytes of traffic --; every
 * other program materialises the same stream into noise_scratch:(B,D) (required then) and runs as b2f_flow_apply.
 * With B2F_FLOW_LOGP_OF_INPUT, log_prob = base density of z + log_det as Flow.sample(return_log_prob=True) returns. */
int b2f_flow_sample(const b2f_op_t *ops, int32_t n_ops, float *y, float *log_det, float *log_prob, const float *base_loc,
                    const float *base_log_scale, float *noise_scratch, int64_t B, int32_t D, int32_t flags, uint64_t seed,
                    uint64_t offset, void *stream);
/* The same stream materialised: out:(n_rows, D) = loc + exp(log_scale) * n  (DiagonalGaussian.sample). */
int b2f_philox_normal(float *out, int64_t n_rows, int32_t D, const float *loc, const float *log_scale, uint64_t seed,
                      uint64_t offset, void *stream);

/* b2f_flow_apply for a training step: additionally writes, for every COUPLING / MADE / MADE_SEQ op in order, the
 * activations as they ENTER that layer into `workspace` ([layer][B][D] floats, b2f_flow_backward_workspace() bytes) --
 * exactly what b2f_flow_backward would otherwise recompute.  *saved = 1 if the kernel that took the program wrote them
 * (today: the tensor-core kernel), 0 if not (the call is then identical to b2f_flow_apply and `workspace` is untouched).
 * With *saved == 1 call b2f_flow_backward with B2F_FLOW_WS_FILLED, the same workspace and x = the OUTPUT y of this call.
 * Replaces the activations torch autograd keeps alive for backward (flows.py:199-224). */
int b2f_flow_apply_saving(const b2f_op_t *ops, int32_t n_ops, const float *x, float *y, float *log_det, float *log_prob,
                          const float *base_loc, const float *base_log_scale, void *workspace, int32_t *saved, int64_t B,
                          int32_t D, int32_t flags, void *stream);
#define B2F_FLOW_WS_FILLED 8 /* b2f_flow_backward: `workspace` already holds the layer inputs (b2f_flow_apply_saving) and
                                `x` is the forward OUTPUT; the forward recompute is skipped */

/* Backward of b2f_flow_apply in the density direction: given the saved input x and upstream gradients
 * gy:(B,D) (nullable), glog_det:(B) (nullable), glog_prob:(B) (nullable), recomputes the forward per tile and
 * produces gx:(B,D) (nullable) and accumulates parameter gradients into ops[i].g[].  Replaces autograd
 * through the same reference code.  `workspace` holds the saved layer inputs: b2f_flow_backward_workspace()
 * bytes. */
int b2f_flow_backward(const b2f_op_t *ops, int32_t n_ops, const float *x, const float *gy, const float *glog_det,
                      const float *glog_prob, const float *base_loc, const float *base_log_scale, float *gx,
                      void *workspace, int64_t B, int32_t D, int32_t flags, void *stream);
int64_t b2f_flow_backward_workspace(const b2f_op_t *ops, int32_t n_ops, int64_t B, int32_t D);
/* 1 if b2f_flow_backward can run this program at event size D (some tile shape of the backward kernel fits shared memory),
 * else 0.  Only kind, tkind, n_hidden and n_bins of the ops are looked at, so callers can ask before any parameter exists
 * (torchflows_b200 decides at construction time whether a layer trains through the fused kernel or as a composite). */
int32_t b2f_flow_backward_fits(const b2f_op_t *ops, int32_t n_ops, int32_t D);
/* The tile shape b2f_flow_backward would launch for this program with these flags: returns 1 and writes out[0] = rows
 * per tile TM, out[1] = threads per CTA NT and out[2] = the per-warp staging stride of a spline layer's output weights
 * in floats (0: spline layers take the scalar GEMM path), or returns 0 if the kernel cannot take the program.  Host-only;
 * honours B2F_FLOW_MODE_PRECISE and the environment overrides B2F_BWD_TM / B2F_BWD_NT / B2F_BWD_NO_MMA exactly as the
 * launch does, so it tells whether a forced shape was admissible and fitted or fell back to the default one.  Looks at
 * kind, tkind and n_hidden of the ops, and at the alignment of p[2] of spline layers (unaligned output weights disable
 * the staging). */
int32_t b2f_flow_backward_shape(const b2f_op_t *ops, int32_t n_ops, int32_t D, int32_t flags, int32_t out[3]);

/* Elementwise transformer given materialised parameters h (TensorTransformer.forward / inverse,
 * transformers/base.py:24-42): x,out:(n_rows, n_event); h:(n_rows, n_event, P) with row stride
 * h_row_stride floats (0 broadcasts one parameter set over all rows, as ElementwiseBijection.prepare_h does,
 * layers_base.py:300-303); log_det:(n_rows) (nullable) = sum over the event; k_out:(n_rows, n_event) int32
 * (nullable, RQ only) = the bin index used, -1 outside the spline bounds. */
int b2f_transformer_apply(int32_t tkind, const float *x, const float *h, float *out, float *log_det,
                          int32_t *k_out, int64_t n_rows, int32_t n_event, int64_t h_row_stride, int32_t n_bins,
                          float boundary, int32_t flags, void *stream);

/* Backward of b2f_transformer_apply: upstream gout:(n_rows,n_event) (nullable), glog_det:(n_rows) (nullable)
 * -> gx:(n_rows,n_event), gh:(n_rows,n_event,P) (dense, row stride n_event*P). */
int b2f_transformer_backward(int32_t tkind, const float *x, const float *h, const float *gout,
                             const float *glog_det, float *gx, float *gh, int64_t n_rows, int32_t n_event,
                             int64_t h_row_stride, int32_t n_bins, float boundary, int32_t flags, void *stream);

/* ---- wide-conditioner spline coupling layer (csrc/b2f_wide.cu) ------------------------------------------------------
 * One CouplingBijection with HalfSplit + FeedForward(n_layers=2, Tanh) + RationalQuadratic(n_bins=8) whose hidden
 * width is too large for the whole-flow kernels (e.g. n_dim = 1024, n_hidden = 1024): layers_base.py:119-163,
 * conditioning/transforms.py:274-307, transformers/spline/rational_quadratic.py:45-200.  Every contraction (forward,
 * recompute, dgrad, wgrad) runs on tcgen05 kind::tf32; the conditioner output h = (B, D/2 * 23) is never written to
 * memory (the spline, or its backward, is the epilogue of the output-layer GEMM reading tensor memory).
 * Parameters in the reference's own layout: W1 (H, D/2), b1 (H), W2 (D/2 * 23, H), b2 (D/2 * 23).
 * Requirements: D % 64 == 0, H % 32 == 0, n_bins == 8; x, y, workspace 16-byte aligned. */
typedef struct b2f_wide_layer {
    int32_t D;        /* event size; the first D/2 columns are the conditioner input, the rest are transformed */
    int32_t H;        /* n_hidden */
    int32_t tkind;    /* B2F_T_RQ_FWD (CouplingBijection.forward) or B2F_T_RQ_INV (.inverse) */
    int32_t n_bins;   /* 8 */
    float boundary;
    int32_t reserved;
    const float *W1, *b1, *W2, *b2;
} b2f_wide_layer_t;

/* Two caller-owned buffers.  `keep`: packed operands and hidden activations of one layer call -- what the backward of the
 * same step can reuse; `scratch`: temporaries of one call (may be shared by all layers of a flow).
 * which = 0: keep bytes, forward only; 1: keep bytes when a backward follows; 2: scratch bytes of the forward; 3: of the backward. */
int64_t b2f_wide_coupling_workspace(int64_t B, int32_t D, int32_t H, int32_t which);

#define B2F_WIDE_FOR_BACKWARD 1 /* forward flag: also lay out the operands the backward needs (keep sized with which = 1) */
#define B2F_WIDE_KEPT 2         /* backward flag: `keep` still holds what the forward (with B2F_WIDE_FOR_BACKWARD, same x, same
                                   parameters) left there; without it the backward rebuilds it from x and the parameters */

/* y:(B,D) = layer(x:(B,D)), log_det:(B) (nullable).  The conditioner output is never stored; the backward recomputes it. */
int b2f_wide_coupling_forward(const b2f_wide_layer_t *layer, const float *x, float *y, float *log_det, int64_t B, void *keep,
                              int64_t keep_bytes, void *scratch, int64_t scratch_bytes, int32_t flags, void *stream);

/* Given the layer INPUT x and upstream gy:(B,D) (nullable), glog_det:(B) (nullable): gx:(B,D) and the parameter gradients
 * gW1, gb1, gW2, gb2 (reference layouts; overwritten, not accumulated).  Replaces autograd through the reference code above. */
int b2f_wide_coupling_backward(const b2f_wide_layer_t *layer, const float *x, const float *gy, const float *glog_det,
                               float *gx, float *gW1, float *gb1, float *gW2, float *gb2, int64_t B, void *keep,
                               int64_t keep_bytes, void *scratch, int64_t scratch_bytes, int32_t flags, void *stream);

/* ---- runs of per-column layers at any event size (csrc/b2f_colrun.cu) -----------------------------------------------
 * ElementwiseAffine / ActNorm with global parameters (autoregressive/layers_base.py:300-318, transformers/linear/
 * affine.py:33-59, layers.py:39-69) and ReversePermutationMatrix (matrix/permutation.py:19-37) in application order
 * compose into y[r, c] = A[c] x[r, s(c)] + C[c]; one pass over the batch instead of one per layer.  Used between layers
 * that are not part of a whole-flow program (the wide coupling layers above). */
#define B2F_COL_AFFINE_FWD 0 /* z = alpha x + v1,  alpha = exp(log(1 - 1e-10) + v0 / 2) + 1e-10   (Affine.forward) */
#define B2F_COL_AFFINE_INV 1 /* x = (z - v1) / alpha                                               (Affine.inverse) */
#define B2F_COL_FLIP 2       /* y[:, c] = x[:, D - 1 - c] */
#define B2F_COL_MAX_OPS 8
typedef struct b2f_colop {
    int32_t kind;
    int32_t reserved;
    const float *value; /* (D, 2): v0, v1 per column (null for FLIP) */
    float *gvalue;      /* b2f_column_run_backward: gradient of `value`, overwritten (nullable: frozen parameters) */
} b2f_colop_t;

/* y:(B,D); log_det_sum: ONE float (nullable) = sum over columns of log A[c], the log-determinant of every row. */
int b2f_column_run_apply(const b2f_colop_t *ops, int32_t n_ops, const float *x, float *y, float *log_det_sum, int64_t B,
                         int32_t D, void *stream);
/* x: the run's input; gy:(B,D); g_log_det_sum: one float (nullable) = sum over rows of dL/dlog_det.  gx:(B,D) and every
 * op's gvalue; scratch: 2*D floats. */
int b2f_column_run_backward(const b2f_colop_t *ops, int32_t n_ops, const float *x, const float *gy, const float *g_log_det_sum,
                            float *gx, float *scratch, int64_t B, int32_t D, void *stream);

/* DiagonalGaussian.log_prob over rows (base_distributions/gaussian.py:46-54) for flows whose layers are not one program
 * (z:(B,D) comes back from the last layer): log_prob:(B); loc / log_scale:(D) nullable = standard normal.  Backward:
 * gz:(B,D) = dL/dz given g_log_prob:(B) (the base parameters are not differentiated: trainable bases stay on torch ops). */
int b2f_gauss_log_prob(const float *z, const float *loc, const float *log_scale, float *log_prob, int64_t B, int32_t D,
                       void *stream);
int b2f_gauss_log_prob_backward(const float *z, const float *loc, const float *log_scale, const float *g_log_prob, float *gz,
                                int64_t B, int32_t D, void *stream);

/* Per-dimension batch statistics for ActNorm's data-dependent initialisation (layers.py:58-68):
 * sum:(D) and sumsq:(D) of x:(B,D), accumulated in fp64 (must be zeroed by the caller). */
int b2f_column_stats(const float *x, double *sum, double *sumsq, int64_t B, int32_t D, void *stream);

/* Parameters per element of a transformer kind, and its padded count PP used by the W2 tile layout. */
int32_t b2f_params_per_element(int32_t tkind, int32_t n_bins);
int32_t b2f_padded_params(int32_t params_per_element);

/* Diagnostic: one tcgen05 (kind::tf32) GEMM tile C[128,N] = A[128,K] * B[N,K]^T through the same descriptor and
 * operand-layout code as the fused coupling kernel; used by the GPU tests to localise tensor-core layout bugs. */
int b2f_debug_umma_gemm(const float *A, const float *B, float *C, int32_t N, int32_t K, void *stream);

const char *b2f_last_error(void);
int32_t b2f_abi_version(void);

/* Diagnostics: which kernel the calling thread's last successful b2f_flow_apply launched (the dispatch is by program
 * shape, see DESIGN.md "Kernels"): the generic FP32 kernel (csrc/b2f_flow.cu), the tcgen05 kernel (csrc/b2f_flow_tc.cu)
 * or the row-per-thread kernel (csrc/b2f_flow_rows.cu).  No reference counterpart. */
#define B2F_KERNEL_NONE 0
#define B2F_KERNEL_GENERIC 1
#define B2F_KERNEL_TC 2
#define B2F_KERNEL_ROWS 3
#define B2F_KERNEL_TCQ 4 /* csrc/b2f_flow_tcq.cu: spline coupling programs laid out with B2F_FLAG_TCQ_OPERANDS */
#define B2F_KERNEL_TCA 5 /* csrc/b2f_flow_tca.cu: affine / shift coupling programs laid out with B2F_FLAG_TCA_OPERANDS */
#define B2F_KERNEL_TCM 6 /* csrc/b2f_flow_tcm.cu: one-pass MADE spline programs laid out with B2F_FLAG_TCM_OPERANDS */
int32_t b2f_last_flow_kernel(void);

#ifdef __cplusplus
}
#endif
#endif /* B2F_H_ */
