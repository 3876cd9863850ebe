// Spline-coupling whole-flow kernel, second generation ("tcq"): CouplingRQNSF-style programs (ElementwiseAffine / ActNorm,
// ReversePermutation, rational-quadratic coupling layers) in ONE persistent launch, the conditioner on tcgen05, the sample
// tile moved by the TMA engine.
//
// Replaces the same reference code as b2f_flow_tc.cu (bijections/base.py:203-232, layers_base.py:119-163,
// transforms.py:293-307, transformers/spline/rational_quadratic.py:45-200, flows.py:628-648); it differs from that
// kernel in how the work is cut (round-1 profile: 544 thread-instructions per spline element, 16 warps meeting on
// every chunk, synchronous tile IO):
//
//  * operands are laid out by torchflows_b200/_tcq.py: elementwise layers and the permutation are folded into
//    per-column affine maps / weight order (no elementwise passes), the output layer produces the 24 "folded" columns
//    of csrc/b2f_rqfast.cuh (~150 issue slots per element);
//  * the 16 epilogue warps form 4 independent groups (4 warps = 128 TMEM lanes each).  A GEMM2 chunk is 2 elements
//    x 24 columns = N 48 and belongs to ONE group: chunk c goes to group c % 4, TMEM buffer (c / 4) % 2 of that group,
//    so a group only ever waits for its own accumulator and hands it back as soon as the columns are in registers;
//  * log-det and base-density partial sums stay in registers across layers; one shared-memory reduction per tile;
//  * full tiles are loaded / stored with cp.async.bulk.tensor (4-D tensor map whose box IS the canonical K-major
//    UMMA operand layout: {k%4, row%8, k/4, row/8}), the ragged last tile by the epilogue warps.
//
// Shared memory (D = 256, H = 17: 201 KB): xt[2] the two halves of the 128-row tile (canonical [128 x D/2] each, both
// the resident activations and the A operand of GEMM1), w1 [32 x D/2], a2 [128 x K2] (tanh(hidden) | 1 | 1 | 0..),
// w2[8] chunk operands [48 x K2] (slot = group + 4 * buffer), red[4][128] float2.
// Tensor memory: D2 slot (g, b) at columns 96 g + 48 b, D1 at 384..415.
#include <cuda.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>

#include "b2f_flow_device.cuh"
#include "b2f_philox.cuh"
#include "b2f_rqfast.cuh"
#include "b2f_umma.cuh"

#ifndef B2F_TCQ_NY
#define B2F_TCQ_NY 0      // heights exponentials taken from the SFU in the fast variant (rest: cubic on the FMA pipe);
                          // measured on Q256: NY = 0 / 2 / 4 / 8 -> 2.39 / 2.42 / 2.44 / 2.58 ms per 2^20-row log_prob
#endif

namespace b2f {

constexpr int kQEpiWarps = 16;
constexpr int kQThreads = (kQEpiWarps + 3) * 32;     // + MMA issuer, weight loader, tile IO
constexpr int kQN1 = 32;                      // UMMA N of GEMM1 (hidden units, padded)
constexpr int kQN2 = 48;                      // UMMA N of a GEMM2 chunk: 2 elements x 24 columns
constexpr int kQSlots = 8;                    // TMEM accumulator slots: (group, buffer)
constexpr int kQRing = 3;                     // W2 ring entries; one entry = one round = 4 chunks (one per group)
constexpr int kQColD1 = 384;
constexpr int kQTmemCols = 512;
constexpr int kQHdr = 8;                      // header ints of a layer blob
constexpr int kQMaxLayers = 12;

struct QLayer {
    const float* blob;
    int H, K2, inverse;
    float boundary;
};

struct QArgs {
    QLayer layers[kQMaxLayers];
    int n_layers, D, flags, n_tiles, use_tma, n_ring;
    long long B;
    const float* x;
    float* y;
    float* log_det;
    float* log_prob;
    const float* prog;      // program blob: [4 ints][4 consts][D x (fin_a, fin_b)][D x (in_a, in_b)]
    // Flow.sample with in-kernel noise (b2f_flow_sample): the input tile is drawn from the Philox stream instead of loaded
    int philox;
    int no_dpoly;           // B2F_TCQ_NO_DPOLY: SFU softplus for the knot derivatives even where delta_poly is admitted
    unsigned long long seed, offset;
    const float* base_loc;          // nullable: standard normal
    const float* base_log_scale;
};

enum { QB_XA_FULL = 0, QB_XB_FULL, QB_EARLY_FREE, QB_TILE_DONE, QB_W1_FULL, QB_W1_EMPTY, QB_A1_READY, QB_D1_FULL, QB_A2_FULL,
       QB_W2_FULL, QB_W2_EMPTY = QB_W2_FULL + kQRing, QB_D2_FULL = QB_W2_EMPTY + kQRing,
       QB_D2_EMPTY = QB_D2_FULL + kQSlots, QB_COUNT = QB_D2_EMPTY + kQSlots };

struct QSmem {
    float* xt[2];
    float* w1;
    float* a2;
    float* w2;          // ring of n_ring round operands [192 x K2], w2stride floats apart
    int w2stride, n_ring;
    float2* red;        // [4][128]
    float* lpin;        // [128]
    uint64_t* bars;
    uint32_t* tmem_ptr;
};

__device__ __forceinline__ void q_epi_sync() { asm volatile("bar.sync 1, %0;" ::"n"(kQEpiWarps * 32) : "memory"); }

__device__ __forceinline__ float q_tf32_rn(float v) {
    uint32_t r;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(v));
    return __uint_as_float(r);
}

// ---- tensor-map TMA (tile load / store) ---------------------------------------------------------------------------------
__device__ __forceinline__ void q_tma_load4(void* dst, const CUtensorMap* map, int c0, int c1, int c2, int c3, uint64_t* bar) {
    asm volatile("cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4, %5}], [%6];"
                 ::"r"(umma::smem_u32(dst)), "l"(map), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(umma::smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void q_tma_store4(const CUtensorMap* map, int c0, int c1, int c2, int c3, const void* src) {
    asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.tile.bulk_group [%0, {%1, %2, %3, %4}], [%5];"
                 ::"l"(map), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(umma::smem_u32(src)) : "memory");
}
__device__ __forceinline__ void q_bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void q_bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void q_bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }

__device__ __forceinline__ int q_hdr(const float* blob, int i) { return __ldg(reinterpret_cast<const int*>(blob) + i); }

// explicit shared-space accesses (32-bit addresses): the tile pointers depend on the per-tile buffer swap, and generic
// pointers would turn into LD.E / ST.E with address-space resolution on the critical path
__device__ __forceinline__ float2 q_lds64(uint32_t a) {
    float2 v;
    asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(v.x), "=f"(v.y) : "r"(a));
    return v;
}
__device__ __forceinline__ void q_sts64(uint32_t a, float2 v) {
    asm volatile("st.shared.v2.f32 [%0], {%1, %2};" ::"r"(a), "f"(v.x), "f"(v.y) : "memory");
}
__device__ __forceinline__ float4 q_lds128(uint32_t a) {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(a));
    return v;
}
__device__ __forceinline__ void q_sts128(uint32_t a, float4 v) {
    asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(a), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}

// v = a * v + b on 4 consecutive columns; p0 = (a0, b0, a1, b1), p1 = (a2, b2, a3, b3)
__device__ __forceinline__ float4 q_affine4(float4 v, float4 p0, float4 p1) {
    v.x = fmaf(v.x, p0.x, p0.y); v.y = fmaf(v.y, p0.z, p0.w);
    v.z = fmaf(v.z, p1.x, p1.y); v.w = fmaf(v.w, p1.z, p1.w);
    return v;
}

// Cooperative pass of the 16 epilogue warps over one half of the tile: x <- a * x + b per column (params: [Dh][2]).
// Warp w owns rows 8w..8w+7, four lanes share a row and stride over its 16-byte column groups.
__device__ __forceinline__ void q_affine_pass(uint32_t half_addr, uint32_t row_off, const float* __restrict__ params, int Dh, int kq) {
#pragma unroll 4
    for (int kc = kq; kc < Dh / 4; kc += 4) {
        const float4 p0 = __ldg(reinterpret_cast<const float4*>(params + 8 * kc));
        const float4 p1 = __ldg(reinterpret_cast<const float4*>(params + 8 * kc + 4));
        const uint32_t a = half_addr + row_off + kc * 128;
        q_sts128(a, q_affine4(q_lds128(a), p0, p1));
    }
}

// One coupling layer's transformer phase for one epilogue thread (row m, group g): its chunks c = g, g + 4, ...
// DPOLY: knot derivatives from rqf::delta_poly.  LD = false (inverse only): the transformed values alone, ld2 and sq untouched.
template <bool INV, bool SAFE, bool DPOLY, bool LD>
__device__ __forceinline__ void q_chunk_loop(const QSmem& s, const float* __restrict__ tp, float boundary, uint32_t tbase,
                                             uint32_t lane_addr, uint32_t tgt_addr, int Dh, int n_chunks, uint32_t cc_base, int m,
                                             int g, int lane, float& ld2, float& sq) {
    static_assert(INV || LD, "the forward direction always feeds a log-density");
    const uint32_t xrow = tgt_addr + (m >> 3) * (Dh * 32) + (m & 7) * 16;       // canon_off(m, 0, Dh)
    for (int c = g; c < n_chunks; c += 4) {
        const uint32_t ccl = cc_base + c, slot = ccl & (kQSlots - 1);
        umma::mbar_wait(&s.bars[QB_D2_FULL + slot], (ccl >> 3) & 1);
        umma::tc_fence_after_sync();
        const uint32_t tcol = tbase + lane_addr + g * (2 * kQN2) + ((c >> 2) & 1) * kQN2;
        float ga[24], gb[24];
        umma::tmem_ld8_nowait<0>(tcol, ga);
        umma::tmem_ld8_nowait<8>(tcol + 8, ga);
        umma::tmem_ld8_nowait<16>(tcol + 16, ga);
        umma::tmem_ld8_nowait<0>(tcol + 24, gb);
        umma::tmem_ld8_nowait<8>(tcol + 32, gb);
        umma::tmem_ld8_nowait<16>(tcol + 40, gb);
        umma::tmem_ld_wait();
        umma::tc_fence_before_sync();
        if (lane == 0) umma::mbar_arrive(&s.bars[QB_D2_EMPTY + slot]);      // the columns are in registers: hand the buffer back
        // elements 2c, 2c + 1 of the target half: adjacent columns, one 8-byte access
        const int e0 = 2 * c;
        const uint32_t px = xrow + (e0 >> 2) * 128 + (e0 & 3) * 4;
        const float2 xv = q_lds64(px);
        const float4 pa = __ldg(reinterpret_cast<const float4*>(tp + e0 * 8));          // pre_a, pre_b, post_a, post_b
        const float2 fa = __ldg(reinterpret_cast<const float2*>(tp + e0 * 8 + 4));      // fin_a, fin_b
        const float4 pb = __ldg(reinterpret_cast<const float4*>(tp + e0 * 8 + 8));
        const float2 fb = __ldg(reinterpret_cast<const float2*>(tp + e0 * 8 + 12));
        float oa, ob, la, lb;
        const float va = fmaf(xv.x, pa.x, pa.y), vb = fmaf(xv.y, pb.x, pb.y);
        if (INV) {
            rqf::inverse<SAFE, B2F_TCQ_NY, DPOLY, LD>(va, ga, boundary, oa, la);
            rqf::inverse<SAFE, B2F_TCQ_NY, DPOLY, LD>(vb, gb, boundary, ob, lb);
        } else {
            rqf::forward<SAFE, B2F_TCQ_NY, DPOLY>(va, ga, boundary, oa, la);
            rqf::forward<SAFE, B2F_TCQ_NY, DPOLY>(vb, gb, boundary, ob, lb);
        }
        const float sa = fmaf(oa, pa.z, pa.w), sb = fmaf(ob, pb.z, pb.w);
        q_sts64(px, make_float2(sa, sb));
        if (!LD) continue;
        const float ta = fmaf(sa, fa.x, fa.y), tb = fmaf(sb, fb.x, fb.y);
        sq = fmaf(ta, ta, sq);
        sq = fmaf(tb, tb, sq);
        ld2 += la + lb;
    }
}

// Tile buffers.  The two halves of a tile live in the two 64 KB buffers xt[0], xt[1]; which half sits in which buffer
// alternates from tile to tile (`swap`), because the next tile is prefetched half by half into whatever the current tile
// releases first: the source half of the LAST layer is dead once that layer's GEMM1 has read it (EARLY_FREE) and receives
// the next tile's FIRST-layer source half; the other half follows when the tile is done (TILE_DONE).
// LD = false: Flow.sample without log_prob -- neither log-det nor log-density is written, so the inverse layers compute the
// transformed values only and the per-tile reduction is skipped.  Launched only on programs whose layers are all inverse.
template <bool LD>
__global__ void __launch_bounds__(kQThreads, 1)
flow_tcq_kernel(const __grid_constant__ QArgs A, const __grid_constant__ CUtensorMap map_x,
                const __grid_constant__ CUtensorMap map_y) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    const int D = A.D, Dh = D >> 1;
    const int tid = threadIdx.x, lane = tid & 31;
    const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);       // warp-uniform by construction: TMEM / barrier addressing
    int K2max = 8;                                                // stays in the uniform datapath
    for (int i = 0; i < A.n_layers; ++i) K2max = max(K2max, A.layers[i].K2);
    QSmem s;
    uint8_t* p = smem_raw;
    s.xt[0] = reinterpret_cast<float*>(p); p += 128 * Dh * 4;
    s.xt[1] = reinterpret_cast<float*>(p); p += 128 * Dh * 4;
    s.w1 = reinterpret_cast<float*>(p); p += kQN1 * Dh * 4;
    s.a2 = reinterpret_cast<float*>(p); p += 128 * K2max * 4;
    s.w2 = reinterpret_cast<float*>(p); p += A.n_ring * 4 * kQN2 * K2max * 4;
    s.w2stride = 4 * kQN2 * K2max;
    s.n_ring = A.n_ring;
    s.red = reinterpret_cast<float2*>(p); p += 4 * 128 * 8;
    s.lpin = reinterpret_cast<float*>(p); p += 128 * 4;
    s.bars = reinterpret_cast<uint64_t*>(p); p += QB_COUNT * 8;
    s.tmem_ptr = reinterpret_cast<uint32_t*>(p);

    if (tid == 0) {
        umma::mbar_init(&s.bars[QB_XA_FULL], 1);
        umma::mbar_init(&s.bars[QB_XB_FULL], 1);
        umma::mbar_init(&s.bars[QB_EARLY_FREE], kQEpiWarps);
        umma::mbar_init(&s.bars[QB_TILE_DONE], kQEpiWarps);
        umma::mbar_init(&s.bars[QB_W1_FULL], 1);
        umma::mbar_init(&s.bars[QB_W1_EMPTY], 1);
        umma::mbar_init(&s.bars[QB_A1_READY], kQEpiWarps);
        umma::mbar_init(&s.bars[QB_D1_FULL], 1);
        umma::mbar_init(&s.bars[QB_A2_FULL], kQEpiWarps);
        for (int i = 0; i < kQRing; ++i) {
            umma::mbar_init(&s.bars[QB_W2_FULL + i], 1);
            umma::mbar_init(&s.bars[QB_W2_EMPTY + i], 1);
        }
        for (int i = 0; i < kQSlots; ++i) {
            umma::mbar_init(&s.bars[QB_D2_FULL + i], 1);
            umma::mbar_init(&s.bars[QB_D2_EMPTY + i], 4);
        }
        umma::fence_barrier_init();
    }
    if (warp == kQEpiWarps) umma::tmem_alloc(s.tmem_ptr, kQTmemCols);
    umma::tc_fence_before_sync();
    __syncthreads();
    umma::tc_fence_after_sync();
    const uint32_t tbase = *s.tmem_ptr;
    const int n_chunks = Dh >> 1;
    const bool want_lp = A.log_prob != nullptr;
    const bool lp_in = want_lp && (A.flags & B2F_FLOW_LOGP_OF_INPUT);
    const int s_first = q_hdr(A.layers[0].blob, 1), s_last = q_hdr(A.layers[A.n_layers - 1].blob, 1);
    const uint32_t swap_step = s_first != s_last ? 1u : 0u;
    const uint32_t xt0 = umma::smem_u32(s.xt[0]), half_bytes = 128u * Dh * 4;       // buffer b starts at xt0 + b * half_bytes

    uint32_t lc = 0;        // coupling layers processed so far (all roles count identically)
    uint32_t cc = 0;        // GEMM2 chunks processed so far (multiple of 8 at every layer boundary)
    uint32_t tc = 0;        // tiles processed so far
    uint32_t swap = 0;      // half h of the current tile lives in buffer h ^ swap
    uint32_t ring = 0, ring_ph = 0;   // W2 ring position and phase (loader and MMA issuer count identically)

    if (warp == kQEpiWarps + 2) {
        // ===================== tile IO (one thread): tensor-map TMA loads, stores and the half-by-half prefetch =====================
        if (lane == 0) {
            auto is_full = [&](int t) { return A.use_tma && ((long long)t * 128 + 128 <= A.B); };
            auto load_half = [&](int t, int h, uint32_t buf, uint64_t* bar) {
                if (is_full(t) && !A.philox) {
                    umma::mbar_arrive_expect_tx(bar, 128u * Dh * 4);
                    q_tma_load4(reinterpret_cast<uint8_t*>(s.xt[0]) + buf * half_bytes, &map_x, 0, 0, h * (Dh / 4), t * 16, bar);
                } else {
                    umma::mbar_arrive(bar);          // ragged tile: the epilogue warps load it themselves once both arrived
                }
            };
            int tile = blockIdx.x;
            if (tile < A.n_tiles) {
                load_half(tile, s_first, s_first, &s.bars[QB_XA_FULL]);
                load_half(tile, 1 - s_first, 1 - s_first, &s.bars[QB_XB_FULL]);
            }
            for (; tile < A.n_tiles; tile += gridDim.x, ++tc) {
                const int next = tile + gridDim.x;
                const bool store = A.y != nullptr && is_full(tile);
                const uint32_t buf_e = s_last ^ swap, buf_r = buf_e ^ 1u;
                umma::mbar_wait_backoff(&s.bars[QB_EARLY_FREE], tc & 1);
                if (store) {
                    q_tma_store4(&map_y, 0, 0, s_last * (Dh / 4), tile * 16, reinterpret_cast<uint8_t*>(s.xt[0]) + buf_e * half_bytes);
                    q_bulk_commit();
                    q_bulk_wait_read();
                }
                if (next < A.n_tiles) load_half(next, s_first, buf_e, &s.bars[QB_XA_FULL]);
                umma::mbar_wait_backoff(&s.bars[QB_TILE_DONE], tc & 1);
                if (store) {
                    q_tma_store4(&map_y, 0, 0, (1 - s_last) * (Dh / 4), tile * 16, reinterpret_cast<uint8_t*>(s.xt[0]) + buf_r * half_bytes);
                    q_bulk_commit();
                    q_bulk_wait_read();
                }
                if (next < A.n_tiles) load_half(next, 1 - s_first, buf_r, &s.bars[QB_XB_FULL]);
                swap ^= swap_step;
            }
            q_bulk_wait_all();
        }
        __syncwarp();
    } else if (warp == kQEpiWarps + 1) {
        // ===================== weight loader (one thread): bulk copies of W1 and of the W2 rounds =====================
        if (lane == 0) {
            for (int tile = blockIdx.x; tile < A.n_tiles; tile += gridDim.x) {
                for (int li = 0; li < A.n_layers; ++li, ++lc) {
                    const QLayer& L = A.layers[li];
                    umma::mbar_wait(&s.bars[QB_W1_EMPTY], (lc & 1) ^ 1);
                    const uint32_t w1_bytes = kQN1 * Dh * 4;
                    umma::mbar_arrive_expect_tx(&s.bars[QB_W1_FULL], w1_bytes);
                    umma::bulk_g2s(s.w1, L.blob + kQHdr, w1_bytes, &s.bars[QB_W1_FULL]);
                    // output layer: one bulk copy per round (4 consecutive chunks = canonical [192 x K2]), ring of n_ring
                    const float* w2g = L.blob + kQHdr + kQN1 * Dh + 32;
                    const uint32_t rd_bytes = 4 * kQN2 * L.K2 * 4;
                    for (int r = 0; r < n_chunks / 4; ++r) {
                        umma::mbar_wait(&s.bars[QB_W2_EMPTY + ring], ring_ph ^ 1);
                        umma::mbar_arrive_expect_tx(&s.bars[QB_W2_FULL + ring], rd_bytes);
                        umma::bulk_g2s(s.w2 + ring * s.w2stride, w2g + (size_t)r * 4 * kQN2 * L.K2, rd_bytes, &s.bars[QB_W2_FULL + ring]);
                        if (++ring == (uint32_t)s.n_ring) { ring = 0; ring_ph ^= 1; }
                    }
                }
            }
        }
        __syncwarp();
    } else if (warp == kQEpiWarps) {
        // ===================== MMA issuer =====================
        // The whole warp runs the (warp-uniform) control flow so that addresses and descriptors stay in uniform registers;
        // one elected lane issues the tcgen05 instructions.  Per MMA this is a 32-bit add on the descriptor's low word: the
        // issuing thread serves 12 MMAs per round and must stay well below the epilogue's ~1800 cycles per round.
        const uint32_t leader = umma::elect_one();
        const uint32_t idesc1 = umma::make_idesc_tf32(128, kQN1), idesc2 = umma::make_idesc_tf32(128, kQN2);
        const uint32_t w1a = umma::smem_u32(s.w1) >> 4, a2a = umma::smem_u32(s.a2) >> 4;
        const uint64_t d1c = umma::make_smem_desc(0, 128, Dh * 32);
        const uint32_t d1_lo = (uint32_t)d1c, d1_hi = (uint32_t)(d1c >> 32);
        for (int tile = blockIdx.x; tile < A.n_tiles; tile += gridDim.x) {
            for (int li = 0; li < A.n_layers; ++li, ++lc) {
                const QLayer& L = A.layers[li];
                const uint32_t src_buf = (uint32_t)q_hdr(L.blob, 1) ^ swap;
                const uint32_t ph = lc & 1;
                umma::mbar_wait(&s.bars[QB_W1_FULL], ph);
                umma::mbar_wait(&s.bars[QB_A1_READY], ph);
                umma::tc_fence_after_sync();
                if (leader) {
                    // GEMM1: D1[128 x 32] = x_src[128 x Dh] * W1c[32 x Dh]^T, one MMA per 8 columns (256 bytes = 16 units)
                    const uint32_t xa = d1_lo + ((xt0 + src_buf * half_bytes) >> 4), wa = d1_lo + w1a;
                    for (int ks = 0; ks < Dh / 8; ++ks)
                        umma::mma_tf32_ss_parts(tbase + kQColD1, xa + ks * 16, d1_hi, wa + ks * 16, d1_hi, idesc1, ks > 0);
                    umma::mma_commit(&s.bars[QB_D1_FULL]);
                    umma::mma_commit(&s.bars[QB_W1_EMPTY]);
                }
                __syncwarp();
                umma::mbar_wait(&s.bars[QB_A2_FULL], ph);
                umma::tc_fence_after_sync();
                const uint64_t d2c = umma::make_smem_desc(0, 128, L.K2 * 32);
                const uint32_t d2_lo = (uint32_t)d2c, d2_hi = (uint32_t)(d2c >> 32);
                const uint32_t a_lo = d2_lo + a2a;
                const int nk = L.K2 / 8;
                const uint32_t grp_units = (kQN2 / 8) * (L.K2 * 32) / 16;      // 6 row groups of the round operand, in 16-byte units
                for (int r = 0; r < n_chunks / 4; ++r, cc += 4) {
                    // round r: chunk 4r + g for group g, TMEM buffer (cc / 4) & 1
                    const uint32_t b = (cc >> 2) & 1, ph2 = (cc >> 3) & 1;
                    umma::mbar_wait(&s.bars[QB_W2_FULL + ring], ring_ph);
                    const uint32_t w_lo = d2_lo + (umma::smem_u32(s.w2 + ring * s.w2stride) >> 4);
#pragma unroll
                    for (uint32_t g = 0; g < 4; ++g) {
                        const uint32_t slot = g + 4 * b;
                        umma::mbar_wait(&s.bars[QB_D2_EMPTY + slot], ph2 ^ 1);
                        umma::tc_fence_after_sync();
                        if (leader) {
                            const uint32_t dcol = tbase + g * (2 * kQN2) + b * kQN2;
                            const uint32_t wg = w_lo + g * grp_units;
#pragma unroll
                            for (int ks = 0; ks < 4; ++ks)
                                if (ks < nk) umma::mma_tf32_ss_parts(dcol, a_lo + ks * 16, d2_hi, wg + ks * 16, d2_hi, idesc2, ks > 0);
                            umma::mma_commit(&s.bars[QB_D2_FULL + slot]);
                        }
                    }
                    if (leader) umma::mma_commit(&s.bars[QB_W2_EMPTY + ring]);
                    __syncwarp();
                    if (++ring == (uint32_t)s.n_ring) { ring = 0; ring_ph ^= 1; }
                }
            }
            swap ^= swap_step;
        }
    } else {
        // ===================== epilogue warps =====================
        const int q = warp & 3, g = warp >> 2;            // TMEM lane quarter, epilogue group
        const int m = q * 32 + lane;                      // row owned in the transformer phase
        const int m8 = warp * 8 + (lane & 7), kq = lane >> 3;   // row / 16-byte column slot in the cooperative passes
        const uint32_t lane_addr = (uint32_t)(q * 32) << 16;
        const float* prog = A.prog;
        const int fin_pass0 = q_hdr(prog, 1), fin_pass1 = q_hdr(prog, 2);
        const float const_ld = __ldg(prog + 4), const_lp = __ldg(prog + 5);
        const float* fin_params = prog + 8;
        const uint32_t row_off = (m8 >> 3) * (Dh * 32) + (m8 & 7) * 16;     // canon_off(m8, 0, Dh)
        for (int tile = blockIdx.x; tile < A.n_tiles; tile += gridDim.x, ++tc) {
            const long long row0 = (long long)tile * 128;
            const int rows = (int)min(128LL, A.B - row0);
            const bool full = A.use_tma && rows == 128;      // the tile leaves through the TMA engine
            const bool tma_in = full && !A.philox;           // ... and arrived through it
            bool have_b = false;                           // waited for the second half of this tile yet?
            umma::mbar_wait(&s.bars[QB_XA_FULL], tc & 1);
            if (!tma_in || lp_in) { umma::mbar_wait(&s.bars[QB_XB_FULL], tc & 1); have_b = true; }
            if (!tma_in) {
                const bool live = m8 < rows;
                if (A.philox) {
                    // base draws of this tile: z = loc + exp(log_scale) n, n = counter-based normals (b2f_philox.cuh); the
                    // noise matrix never exists in memory (gaussian.py:41-44 + flows.py:693 of the reference)
                    const unsigned long long g0 = (unsigned long long)(row0 + m8) * (unsigned long long)(D / 4);
                    // D / 16 >= 2 independent Philox chains per thread: unrolled so that their 10 dependent rounds overlap
#pragma unroll 4
                    for (int kc = kq; kc < D / 4; kc += 4) {
                        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
                        if (live) {
                            v = philox::normal4(g0 + kc, A.seed, A.offset);
                            if (A.base_log_scale) {
                                const float4 ls = __ldg(reinterpret_cast<const float4*>(A.base_log_scale) + kc);
                                v.x *= __expf(ls.x); v.y *= __expf(ls.y); v.z *= __expf(ls.z); v.w *= __expf(ls.w);
                            }
                            if (A.base_loc) {
                                const float4 lc = __ldg(reinterpret_cast<const float4*>(A.base_loc) + kc);
                                v.x += lc.x; v.y += lc.y; v.z += lc.z; v.w += lc.w;
                            }
                        }
                        const uint32_t hf = (4 * kc) >= Dh, k4 = kc - hf * (Dh / 4);
                        q_sts128((xt0 + (hf ^ swap) * half_bytes) + row_off + k4 * 128, v);
                    }
                } else {
                    const float4* src = reinterpret_cast<const float4*>(A.x + (row0 + m8) * D);
                    for (int kc = kq; kc < D / 4; kc += 4) {
                        const float4 v = live ? __ldg(src + kc) : make_float4(0.f, 0.f, 0.f, 0.f);
                        const uint32_t hf = (4 * kc) >= Dh, k4 = kc - hf * (Dh / 4);
                        q_sts128((xt0 + (hf ^ swap) * half_bytes) + row_off + k4 * 128, v);
                    }
                }
                q_epi_sync();
            }
            if (lp_in) {
                // Flow.sample(return_log_prob=True): base density of the INPUT rows (flows.py:710-712)
                const float* ip = prog + 8 + 2 * D;
                float acc = 0.0f;
                for (int kc = kq; kc < D / 4; kc += 4) {
                    const uint32_t hf = (4 * kc) >= Dh, k4 = kc - hf * (Dh / 4);
                    const float4 v = q_lds128((xt0 + (hf ^ swap) * half_bytes) + row_off + k4 * 128);
                    const float4 p0 = __ldg(reinterpret_cast<const float4*>(ip + 8 * kc));
                    const float4 p1 = __ldg(reinterpret_cast<const float4*>(ip + 8 * kc + 4));
                    const float4 t = q_affine4(v, p0, p1);
                    acc = fmaf(t.x, t.x, acc); acc = fmaf(t.y, t.y, acc); acc = fmaf(t.z, t.z, acc); acc = fmaf(t.w, t.w, acc);
                }
                acc += __shfl_xor_sync(0xffffffffu, acc, 8);
                acc += __shfl_xor_sync(0xffffffffu, acc, 16);
                if (kq == 0) s.lpin[m8] = acc;
            }
            float ld2 = 0.0f, sq = 0.0f;
            for (int li = 0; li < A.n_layers; ++li, ++lc) {
                const QLayer& L = A.layers[li];
                const float* blob = L.blob;
                const int src_half = q_hdr(blob, 1), src_pass = q_hdr(blob, 2);
                const uint32_t src_addr = xt0 + ((uint32_t)src_half ^ swap) * half_bytes, tgt_addr = xt0 + ((uint32_t)src_half ^ swap ^ 1u) * half_bytes;
                const int H = L.H, K2 = L.K2;
                const float* b1 = blob + kQHdr + kQN1 * Dh;
                const float* tp = b1 + 32 + (size_t)n_chunks * kQN2 * K2;
                const float* sp = tp + Dh * 8;
                const float* misc = sp + Dh * 2;
                if (src_pass) {
                    // the elementwise layers in front of this layer, applied to the half that feeds the conditioner
                    if (li > 0) {
                        if (!have_b) { umma::mbar_wait(&s.bars[QB_XB_FULL], tc & 1); have_b = true; }
                        q_epi_sync();
                    }
                    q_affine_pass(src_addr, row_off, sp, Dh, kq);
                }
                umma::fence_proxy_async_smem();            // generic-proxy writes to the tile -> tensor core
                __syncwarp();
                if (lane == 0) umma::mbar_arrive(&s.bars[QB_A1_READY]);
                // hidden layer: D1 -> + b1 -> tanh -> tf32 -> a2; group g owns hidden units 8g .. 8g+7, columns H, H+1 are
                // the constant 1 that multiplies the (hi, lo) split of the output bias, the rest of K2 is zero
                umma::mbar_wait(&s.bars[QB_D1_FULL], lc & 1);
                umma::tc_fence_after_sync();
                if (8 * g < K2) {
                    float v[8];
                    umma::tmem_ld8(tbase + lane_addr + kQColD1 + 8 * g, v);
                    umma::tmem_ld_wait();
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                        const int j = 8 * g + i;
                        if (j < H) {
                            const float e = rqf::f_ex2((v[i] + __ldg(b1 + j)) * (2.0f * rqf::kLog2e));
                            v[i] = q_tf32_rn(1.0f - 2.0f * rqf::f_rcp(1.0f + e));       // tanh
                        } else {
                            v[i] = (j < H + 2) ? 1.0f : 0.0f;
                        }
                    }
                    const uint32_t a2row = umma::smem_u32(s.a2) + (m >> 3) * (K2 * 32) + (m & 7) * 16 + (2 * g) * 128;
                    q_sts128(a2row, make_float4(v[0], v[1], v[2], v[3]));
                    q_sts128(a2row + 128, make_float4(v[4], v[5], v[6], v[7]));
                }
                umma::tc_fence_before_sync();
                umma::fence_proxy_async_smem();
                __syncwarp();
                if (lane == 0) umma::mbar_arrive(&s.bars[QB_A2_FULL]);
                if (li == A.n_layers - 1) {
                    // GEMM1 of the last layer has read its source half for the last time: bring it to its final value (sampling:
                    // the elementwise layers still pending on it) and release it -- it is stored and refilled with the next
                    // tile's first half while this layer's transformer phase runs
                    if (A.y && (src_half ? fin_pass1 : fin_pass0)) q_affine_pass(src_addr, row_off, fin_params + src_half * Dh * 2, Dh, kq);
                    umma::fence_proxy_async_smem();
                    __syncwarp();
                    if (lane == 0) umma::mbar_arrive(&s.bars[QB_EARLY_FREE]);
                }
                if (!have_b) { umma::mbar_wait(&s.bars[QB_XB_FULL], tc & 1); have_b = true; }
                // transformer phase.  misc[2] = 0 means no bound on the derivative logits (it is never 0 otherwise: it
                // includes the padded edge logit)
                const bool fast = __ldg(misc) < rqf::kNoMaxBound && __ldg(misc + 1) < rqf::kPolyBound;
                const float bound_d = __ldg(misc + 2);
                const bool dpoly = fast && !A.no_dpoly && bound_d > 0.0f && bound_d < rqf::kDeltaPolyBound;
#define B2F_Q_CHUNKS(INV, SAFE, DPOLY, LDV) \
    q_chunk_loop<INV, SAFE, DPOLY, LDV>(s, tp, L.boundary, tbase, lane_addr, tgt_addr, Dh, n_chunks, cc, m, g, lane, ld2, sq)
                if (LD && !L.inverse) {
                    if (dpoly) B2F_Q_CHUNKS(false, false, true, true);
                    else if (fast) B2F_Q_CHUNKS(false, false, false, true);
                    else B2F_Q_CHUNKS(false, true, false, true);
                } else {
                    if (dpoly) B2F_Q_CHUNKS(true, false, true, LD);
                    else if (fast) B2F_Q_CHUNKS(true, false, false, LD);
                    else B2F_Q_CHUNKS(true, true, false, LD);
                }
#undef B2F_Q_CHUNKS
                cc += n_chunks;
            }
            // ---- outputs of this tile ----
            if (LD) s.red[g * 128 + m] = make_float2(ld2, sq);
            q_epi_sync();                         // also orders the last layer's writes before the passes over the tile
            if (LD && tid < 128) {
                const float2 r0 = s.red[tid], r1 = s.red[128 + tid], r2 = s.red[256 + tid], r3 = s.red[384 + tid];
                const float ld = fmaf((r0.x + r1.x) + (r2.x + r3.x), rqf::kLn2, const_ld);
                float sqs = (r0.y + r1.y) + (r2.y + r3.y);
                if (lp_in) sqs = s.lpin[tid];
                if (tid < rows) {
                    if (A.log_det) A.log_det[row0 + tid] = ld;
                    if (want_lp) A.log_prob[row0 + tid] = fmaf(-0.5f, sqs, const_lp) + ld;
                }
            }
            if (A.y) {
                // the half the last layer wrote: elementwise layers still pending at the end of the program, then out
                const uint32_t hf = 1 - s_last;
                if (hf ? fin_pass1 : fin_pass0) q_affine_pass((xt0 + (hf ^ swap) * half_bytes), row_off, fin_params + hf * Dh * 2, Dh, kq);
                if (!full) {
                    q_epi_sync();
                    if (m8 < rows) {
                        float4* dst = reinterpret_cast<float4*>(A.y + (row0 + m8) * D);
                        for (int kc = kq; kc < D / 4; kc += 4) {
                            const uint32_t h2 = (4 * kc) >= Dh, k4 = kc - h2 * (Dh / 4);
                            dst[kc] = q_lds128((xt0 + (h2 ^ swap) * half_bytes) + row_off + k4 * 128);
                        }
                    }
                }
            }
            umma::fence_proxy_async_smem();       // our accesses to the tile are ordered before the TMA store / the next tile's TMA writes
            __syncwarp();
            if (lane == 0) umma::mbar_arrive(&s.bars[QB_TILE_DONE]);
            swap ^= swap_step;
        }
    }
    umma::tc_fence_before_sync();
    __syncthreads();
    if (warp == kQEpiWarps) umma::tmem_dealloc(tbase, kQTmemCols);
}

// ---- host side --------------------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_tiled_fn() {
    static EncodeTiledFn fn = []() -> EncodeTiledFn {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) != cudaSuccess ||
            qres != cudaDriverEntryPointSuccess)
            return nullptr;
        return reinterpret_cast<EncodeTiledFn>(p);
    }();
    return fn;
}

// (B, D) fp32 row-major seen as {k % 4, row % 8, k / 4, row / 8}; one box = one half of a 128-row tile, written to shared
// memory in exactly the canonical K-major operand order of b2f_umma.cuh.
static bool make_tile_map(CUtensorMap* map, const float* base, long long B, int D) {
    EncodeTiledFn fn = encode_tiled_fn();
    if (!fn || B < 128) return false;
    const cuuint64_t gdim[4] = {4, 8, (cuuint64_t)(D / 4), (cuuint64_t)(B / 8)};
    const cuuint64_t gstride[3] = {(cuuint64_t)D * 4, 16, (cuuint64_t)D * 32};
    const cuuint32_t box[4] = {4, 8, (cuuint32_t)(D / 8), 16};
    const cuuint32_t estr[4] = {1, 1, 1, 1};
    return fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, const_cast<float*>(base), gdim, gstride, box, estr,
              CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
              CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// Returns 1 if the kernel was launched, 0 if the program is not for this kernel (caller falls through), < 0 on error.
int try_launch_flow_tcq(const b2f_op_t* ops, int32_t n_ops, const float* x, float* y, float* log_det, float* log_prob,
                        int64_t B, int32_t D, int32_t flags, void* stream, const TcqNoise* noise) {
    if (getenv("B2F_DISABLE_TCQ") || getenv("B2F_DISABLE_TC") || (flags & B2F_FLOW_MODE_PRECISE)) return 0;
    if (D % 32 != 0 || D < 32 || D > 256) return 0;
    if ((!noise && (reinterpret_cast<uintptr_t>(x) & 15)) || (y && (reinterpret_cast<uintptr_t>(y) & 15))) return 0;
    if (noise && ((reinterpret_cast<uintptr_t>(noise->base_loc) | reinterpret_cast<uintptr_t>(noise->base_log_scale)) & 15)) return 0;
    QArgs A;
    memset(&A, 0, sizeof(A));
    int flip = 0, K2max = 8;
    const float* prog = nullptr;
    for (int i = 0; i < n_ops; ++i) {
        const b2f_op_t& o = ops[i];
        if (o.kind == B2F_OP_FLIP) { flip ^= 1; continue; }
        if (o.kind == B2F_OP_ELEMENTWISE && (o.flags & B2F_FLAG_ROW_BIAS)) return 0;      // per-row parameters: generic kernel
        if (o.kind == B2F_OP_ELEMENTWISE) continue;                 // folded into the blobs by the caller
        if (o.kind != B2F_OP_COUPLING || !(o.flags & B2F_FLAG_TCQ_OPERANDS)) return 0;
        if (o.flags & B2F_FLAG_ROW_BIAS) return 0;
        if ((o.tkind != B2F_T_RQ_FWD && o.tkind != B2F_T_RQ_INV) || o.n_bins != 8) return 0;
        if (o.n_hidden < 1 || o.n_hidden > 30 || !o.p[4] || A.n_layers >= kQMaxLayers) return 0;
        if (reinterpret_cast<uintptr_t>(o.p[4]) & 15)
            return fail(B2F_ERR_INVALID, "op %d: tcq operand blob must be 16-byte aligned", i);
        if (!prog) prog = (const float*)o.p[5];
        QLayer& L = A.layers[A.n_layers++];
        L.blob = (const float*)o.p[4];
        L.H = o.n_hidden;
        L.K2 = (o.n_hidden + 2 + 7) / 8 * 8;
        L.inverse = o.tkind == B2F_T_RQ_INV;
        L.boundary = o.boundary;
        if (!(o.boundary > 0.0f)) return fail(B2F_ERR_INVALID, "op %d: boundary", i);
        K2max = std::max(K2max, L.K2);
    }
    if (flip != 0 || A.n_layers == 0 || !prog) return 0;
    const int Dh = D / 2;
    auto smem_bytes = [&](int n_ring) {
        return (size_t)2 * 128 * Dh * 4 + (size_t)kQN1 * Dh * 4 + (size_t)128 * K2max * 4 +
               (size_t)n_ring * 4 * kQN2 * K2max * 4 + 4 * 128 * 8 + 128 * 4 + QB_COUNT * 8 + 16;
    };
    A.n_ring = kQRing;
    while (A.n_ring > 2 && smem_bytes(A.n_ring) > 227 * 1024) --A.n_ring;
    const size_t smem = smem_bytes(A.n_ring);
    if (smem > 227 * 1024) return 0;
    A.D = D; A.flags = flags; A.B = B;
    A.n_tiles = (int)((B + 127) / 128);
    A.x = x; A.y = y; A.log_det = log_det; A.log_prob = log_prob; A.prog = prog;
    CUtensorMap map_x, map_y;
    memset(&map_x, 0, sizeof(map_x));
    memset(&map_y, 0, sizeof(map_y));
    A.use_tma = getenv("B2F_TCQ_NO_TMA") ? 0 : 1;
    if (noise) {
        A.philox = 1; A.seed = noise->seed; A.offset = noise->offset;
        A.base_loc = noise->base_loc; A.base_log_scale = noise->base_log_scale;
    }
    if (A.use_tma && !noise && !make_tile_map(&map_x, x, B, D)) A.use_tma = 0;
    if (A.use_tma && y && !make_tile_map(&map_y, y, B, D)) A.use_tma = 0;
    A.no_dpoly = getenv("B2F_TCQ_NO_DPOLY") ? 1 : 0;
    // the output-only kernel when nothing reads the log-det (Flow.sample without log_prob) and every layer is inverse
    bool ld = log_det || log_prob || getenv("B2F_TCQ_ALWAYS_LD");
    for (int i = 0; i < A.n_layers; ++i) ld = ld || !A.layers[i].inverse;
    int dev = 0, n_sm = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev);
    const int grid = std::min(A.n_tiles, n_sm);
    const void* kfn = ld ? (const void*)flow_tcq_kernel<true> : (const void*)flow_tcq_kernel<false>;
    cudaError_t ce = (cudaError_t)raise_smem_limit(kfn, smem);
    if (ce != cudaSuccess) return fail(B2F_ERR_CUDA, "cudaFuncSetAttribute(tcq): %s", cudaGetErrorString(ce));
    if (ld) flow_tcq_kernel<true><<<grid, kQThreads, smem, (cudaStream_t)stream>>>(A, map_x, map_y);
    else flow_tcq_kernel<false><<<grid, kQThreads, smem, (cudaStream_t)stream>>>(A, map_x, map_y);
    const int rc = check_launch("b2f_flow_apply (spline tensor-core kernel)");
    return rc == B2F_OK ? 1 : rc;
}

}  // namespace b2f
