// kfpos_score.cu -- scores the ranging selection of a replay (T6) or an ML batch against the NLOS truth of the
// ranging generator (kfpos_batch_score_selection, DESIGN §4.5d).
//
// One thread per (filter, row): the M rangings of its epoch give the present set (the replay's rule of
// convert_epoch: value > 0), `sel` gives the used set, `nlos` the biased rangings.  Every load is coalesced along
// the filter index.  The eight counts of a row are integers, summed in the warp with __reduce_add_sync, then over
// the block in shared memory, then with one 64-bit atomic per block, column and row: the result does not depend on
// the launch geometry or on the order of the atomics.  The kernel is bound by HBM (it reads the log once).
#include "kfpos_kernels.cuh"

namespace kfpos {

namespace {

constexpr int SCORE_BLOCK = 256;
constexpr int SCORE_WARPS = SCORE_BLOCK / 32;

template <int FMT>
__global__ void __launch_bounds__(SCORE_BLOCK) score_selection_kernel(const ScoreParams p) {
    __shared__ unsigned part[SCORE_WARPS][SCORE_COLS];
    const int64_t N = p.N, r = blockIdx.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int64_t fb = blockIdx.y; fb * SCORE_BLOCK < N; fb += gridDim.y) {
        const int64_t f = fb * SCORE_BLOCK + threadIdx.x;
        unsigned c[SCORE_COLS] = {0u, 0u, 0u, 0u, 0u, 0u, 0u, 0u};
        if (f < N) {
            const unsigned present = present_mask<FMT>(p.ranges, r * p.M * N + f, p.M, N);
            const unsigned used = used_mask(present, p.sel, r, N, f, p.mode);
            const unsigned dropped = present & ~used;
            const unsigned nl = p.nlos ? __ldg(p.nlos + r * N + f) & present : 0u;
            c[0] = __popc(present);
            c[1] = __popc(dropped);
            c[2] = __popc(nl);
            c[3] = __popc(nl & dropped);
            c[4] = nl != 0u;
            c[5] = nl != 0u && (nl & used) == 0u;
            c[6] = dropped != 0u;
            c[7] = dropped != 0u && nl == 0u;
        }
#pragma unroll
        for (int q = 0; q < SCORE_COLS; ++q) c[q] = __reduce_add_sync(0xffffffffu, c[q]);
        if (lane < SCORE_COLS) part[warp][lane] = c[lane];
        __syncthreads();
        if (threadIdx.x < SCORE_COLS) {
            unsigned long long s = 0;
#pragma unroll
            for (int w = 0; w < SCORE_WARPS; ++w) s += part[w][threadIdx.x];
            if (s) atomicAdd(p.counts + r * SCORE_COLS + threadIdx.x, s);
        }
        __syncthreads(); // `part` is reused by the next filter block
    }
}

} // namespace

cudaError_t launch_score_selection(const ScoreParams &p, cudaStream_t s) {
    if (p.N <= 0 || p.n_rows <= 0) return cudaSuccess;
    // rows along x, the fastest block index: the blocks resident at one time add into the counters of many rows,
    // not all into the eight of one row
    const int64_t blocks = (p.N + SCORE_BLOCK - 1) / SCORE_BLOCK;
    const dim3 grid((unsigned)p.n_rows, (unsigned)(blocks < 65535 ? blocks : 65535));
    switch (p.fmt) {
    case 0: score_selection_kernel<0><<<grid, SCORE_BLOCK, 0, s>>>(p); break;
    case 1: score_selection_kernel<1><<<grid, SCORE_BLOCK, 0, s>>>(p); break;
    default: score_selection_kernel<2><<<grid, SCORE_BLOCK, 0, s>>>(p); break;
    }
    return cudaGetLastError();
}

} // namespace kfpos
