// Row-per-thread whole-flow kernel, instantiations for programs with sequential spline layers
// (MaskedAutoregressiveRQNSF / MaskedAutoregressiveLRS sampling, InverseAutoregressiveRQNSF / InverseAutoregressiveLRS density): device code in b2f_flow_rows.cuh
// (rows_sequential_rq), eligibility and launch geometry in b2f_flow_rows.cu.  A separate translation unit only to
// compile the spline variants in parallel with the affine ones.
#include "b2f_flow_rows.cuh"

namespace b2f {

template <int MODE>
static cudaError_t launch_spline_h(int hp4, const RowsArgs& A, unsigned grid, size_t smem, cudaStream_t st) {
    switch (hp4) {
        case 1: return launch_rows_kernel<MODE, 1, true, kRowsThreadsSpline>(A, grid, smem, st);
        case 2: return launch_rows_kernel<MODE, 2, true, kRowsThreadsSpline>(A, grid, smem, st);
        case 3: return launch_rows_kernel<MODE, 3, true, kRowsThreadsSpline>(A, grid, smem, st);
        default: return launch_rows_kernel<MODE, 4, true, kRowsThreadsSpline>(A, grid, smem, st);
    }
}

cudaError_t launch_rows_spline(int mode, int hp4, const RowsArgs& A, unsigned grid, size_t smem, cudaStream_t st) {
    // default and fast arithmetic; `precise` programs stay on the generic kernel (b2f_flow_rows.cu does not send them here)
    return mode == 2 ? launch_spline_h<2>(hp4, A, grid, smem, st) : launch_spline_h<1>(hp4, A, grid, smem, st);
}

}  // namespace b2f
