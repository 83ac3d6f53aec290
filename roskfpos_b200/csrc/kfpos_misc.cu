// kfpos_misc.cu -- layout conversion and statistics kernels.
#include "kfpos_kernels.cuh"

namespace kfpos {

// full row-major [n*n][N] -> packed lower triangle [n(n+1)/2][N].  The reference
// covariance is symmetric up to rounding; the lower triangle is kept.
__global__ void pack_cov_kernel(int n, int64_t N, const double *full, double *packed) {
    const int64_t f = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= N) return;
    int k = 0;
    for (int i = 0; i < n; ++i)
        for (int j = 0; j <= i; ++j, ++k) packed[(int64_t)k * N + f] = full[(int64_t)(i * n + j) * N + f];
}

__global__ void unpack_cov_kernel(int n, int64_t N, const double *packed, double *full) {
    const int64_t f = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= N) return;
    int k = 0;
    for (int i = 0; i < n; ++i)
        for (int j = 0; j <= i; ++j, ++k) {
            const double v = packed[(int64_t)k * N + f];
            full[(int64_t)(i * n + j) * N + f] = v;
            full[(int64_t)(j * n + i) * N + f] = v;
        }
}

cudaError_t launch_pack_cov(int n, int64_t N, const double *full, double *packed, cudaStream_t s) {
    if (N <= 0) return cudaSuccess;
    pack_cov_kernel<<<(unsigned)((N + 255) / 256), 256, 0, s>>>(n, N, full, packed);
    return cudaGetLastError();
}

cudaError_t launch_unpack_cov(int n, int64_t N, const double *packed, double *full, cudaStream_t s) {
    if (N <= 0) return cudaSuccess;
    unpack_cov_kernel<<<(unsigned)((N + 255) / 256), 256, 0, s>>>(n, N, packed, full);
    return cudaGetLastError();
}

// ---- error statistics (summation order: kfpos_kernels.cuh, block_stats_partial)
__global__ void __launch_bounds__(STATS_CHUNK)
error_stats_chunks(int64_t N, const double *x, int zrow, double zconst, const int32_t *status, const double *truth,
                   double *partials) {
    __shared__ double sh[4 * STATS_CHUNK];
    double v[4] = {0, 0, 0, 0};
    const int64_t f = (int64_t)blockIdx.x * STATS_CHUNK + threadIdx.x;
    if (f < N) {
        const double pz = zrow >= 0 ? x[(int64_t)zrow * N + f] : zconst;
        filter_error_terms(x[f], x[N + f], pz, truth, N, f, status && status[f] != 0, v);
    }
    block_stats_partial(v, sh, partials + (int64_t)blockIdx.x * 4);
}

// pairwise tree over the partial index, one block per row: the same shape whatever produced the partials.
// The first level reads `src` (src == part: in place); an element left without a partner there is copied.
template <int W>
__global__ void __launch_bounds__(1024) error_stats_tree(int64_t n, const double *src, double *part, int64_t row_stride,
                                                         int64_t es, double *out) {
    src += (int64_t)blockIdx.x * row_stride;
    part += (int64_t)blockIdx.x * row_stride;
    out += (int64_t)blockIdx.x * W;
    if (src != part && (n & 1) && threadIdx.x == 0) {
#pragma unroll
        for (int q = 0; q < W; ++q) part[(n - 1) * es + q] = src[(n - 1) * es + q];
    }
    for (int64_t stride = 1; stride < n; stride <<= 1) {
        const double *in = stride == 1 ? src : part;
        for (int64_t i = (int64_t)threadIdx.x * 2 * stride; i + stride < n; i += (int64_t)blockDim.x * 2 * stride) {
#pragma unroll
            for (int q = 0; q < W; ++q) part[i * es + q] = in[i * es + q] + in[(i + stride) * es + q];
        }
        __syncthreads();
    }
    if (threadIdx.x < W) out[threadIdx.x] = n > 0 ? (n > 1 ? part : src)[threadIdx.x] : 0.0;
}

__global__ void i32_to_f64_kernel(int64_t N, const int32_t *in, double *out) {
    const int64_t f = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (f < N) out[f] = (double)in[f];
}

cudaError_t launch_i32_to_f64(int64_t N, const int32_t *in, double *out, cudaStream_t s) {
    if (N <= 0) return cudaSuccess;
    i32_to_f64_kernel<<<(unsigned)((N + 255) / 256), 256, 0, s>>>(N, in, out);
    return cudaGetLastError();
}

cudaError_t launch_error_stats(int64_t N, const double *x, int zrow, double zconst, const int32_t *status,
                               const double *truth, double *partials, double *out4, cudaStream_t s) {
    const int64_t n_chunks = (N + STATS_CHUNK - 1) / STATS_CHUNK;
    if (n_chunks > 0 && truth)
        error_stats_chunks<<<(unsigned)n_chunks, STATS_CHUNK, 0, s>>>(N, x, zrow, zconst, status, truth, partials);
    return launch_error_stats_tree(n_chunks, partials, out4, s);
}

cudaError_t launch_error_stats_tree(int64_t n, double *part, double *out4, cudaStream_t s) {
    return launch_stats_tree(4, 1, n, part, part, 0, 4, out4, s);
}

cudaError_t launch_stats_tree(int width, int64_t rows, int64_t n, const double *src, double *part, int64_t row_stride,
                              int64_t elem_stride, double *out, cudaStream_t s) {
    if (rows <= 0) return cudaSuccess;
    if (rows > 0x7fffffffLL) return cudaErrorInvalidValue;
    if (width == 4) error_stats_tree<4><<<(unsigned)rows, 1024, 0, s>>>(n, src, part, row_stride, elem_stride, out);
    else if (width == ES_W) error_stats_tree<ES_W><<<(unsigned)rows, 1024, 0, s>>>(n, src, part, row_stride, elem_stride, out);
    else return cudaErrorInvalidValue;
    return cudaGetLastError();
}


// ---- FP64 roofline denominator: a DFMA-only kernel (8 independent chains per
// thread, 2 resident 256-thread blocks per SM-quarter) timed with CUDA events.
__global__ void __launch_bounds__(256) fp64_peak_kernel(double *out, int iters, double a, double b) {
    double v0 = threadIdx.x, v1 = v0 + 1, v2 = v0 + 2, v3 = v0 + 3, v4 = v0 + 4, v5 = v0 + 5, v6 = v0 + 6, v7 = v0 + 7;
    for (int i = 0; i < iters; ++i) {
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            v0 = fma(v0, a, b); v1 = fma(v1, a, b); v2 = fma(v2, a, b); v3 = fma(v3, a, b);
            v4 = fma(v4, a, b); v5 = fma(v5, a, b); v6 = fma(v6, a, b); v7 = fma(v7, a, b);
        }
    }
    const double r = ((v0 + v1) + (v2 + v3)) + ((v4 + v5) + (v6 + v7));
    if (r == 12345.678) out[0] = r; // never true: keeps the chains alive
}

cudaError_t measure_fp64_peak(double *flops_per_s) {
    cudaDeviceProp prop;
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    if ((e = cudaGetDeviceProperties(&prop, dev)) != cudaSuccess) return e;
    double *d = nullptr;
    if ((e = cudaMalloc(&d, sizeof(double))) != cudaSuccess) return e;
    cudaEvent_t t0, t1;
    cudaEventCreate(&t0);
    cudaEventCreate(&t1);
    const int blocks = prop.multiProcessorCount * 8, iters = 4096;
    double best = 0.0;
    for (int rep = 0; rep < 6; ++rep) {
        cudaEventRecord(t0);
        fp64_peak_kernel<<<blocks, 256>>>(d, iters, 0.999999, 1e-9);
        cudaEventRecord(t1);
        if ((e = cudaEventSynchronize(t1)) != cudaSuccess) break;
        float ms = 0;
        cudaEventElapsedTime(&ms, t0, t1);
        const double flops = 2.0 * 64.0 * iters * 256.0 * blocks;
        if (rep > 0 && ms > 0 && flops / (ms * 1e-3) > best) best = flops / (ms * 1e-3);
    }
    cudaEventDestroy(t0);
    cudaEventDestroy(t1);
    cudaFree(d);
    *flops_per_s = best;
    return e;
}

// stateToPose of the three filters (TOA.cpp:159-183, KF.cpp:324-363, TOAIMU.cpp:198-241) on the
// predicted state / covariance of getPose, laid out the way the publisher reads a report
// (Posgenerator.cpp:385-470): pose SoA [13][N] = x, y, z, rotX, rotY, rotZ, rotW, linearSpeed(3),
// angularSpeed(3); cov SoA [36][N], cov[i] = covarianceMatrix(i), Armadillo's column-major index.
// x: SoA [n][N] predicted state; Pf: SoA [n*n][N] predicted covariance, row-major.
__global__ void pose_msg_kernel(int model, int64_t N, double tag_z, const double *tagz, const double *x,
                                const double *Pf, double *pose, double *cov) {
    const int64_t f = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= N) return;
    if (tagz) tag_z = tagz[f]; // per-filter tag height (K8 after a 3-D ML initialisation)
    const int n = model == 1 ? 6 : (model == 2 ? 8 : 9);
    auto X = [&](int i) { return x[(int64_t)i * N + f]; };
    auto P = [&](int i, int j) { return Pf[(int64_t)(i * n + j) * N + f]; };
    double v[13];
#pragma unroll
    for (int i = 0; i < 13; ++i) v[i] = 0.0;
    if (model == 1) {
        v[0] = X(0); v[1] = X(1); v[2] = X(2);
    } else if (model == 2) {
        double sn, cs;
        sincos(X(6) * 0.5, &sn, &cs);
        v[0] = X(0); v[1] = X(1); v[2] = tag_z;
        v[5] = sn; v[6] = cs;
        v[7] = X(2); v[8] = X(3);
        v[12] = X(7);
    } else {
#pragma unroll
        for (int i = 0; i < 3; ++i) {
            v[i] = X(i);
            v[7 + i] = X(3 + i);
            v[10 + i] = X(6 + i); // the acceleration, in the angular-speed fields (TOAIMU.cpp:213-215)
        }
    }
    if (pose) {
#pragma unroll
        for (int i = 0; i < 13; ++i) pose[(int64_t)i * N + f] = v[i];
    }
    if (!cov) return;
    const int nc = model == 3 ? 9 : 6; // dimension of the report's covarianceMatrix
    for (int i = 0; i < 36; ++i) {
        const int r = i % nc, c = i / nc; // column-major linear index
        double val = (r == c && model != 1) ? 0.01 : 0.0;
        if (model == 1) {
            if (r < 3 && c < 3) val = P(r, c);
        } else if (model == 2) {
            const int pr = r == 5 ? 6 : r, pc = c == 5 ? 6 : c; // theta sits in slot 5 of the report
            const bool rs = r < 2 || r == 5, cs2 = c < 2 || c == 5;
            if (rs && cs2) val = P(pr, pc);
        } else {
            const int pr = r == 7 ? 8 : r, pc = c == 7 ? 8 : c;
            const bool rs = r < 3 || r == 7, cs2 = c < 3 || c == 7;
            if (rs && cs2) val = P(pr, pc);
        }
        cov[(int64_t)i * N + f] = val;
    }
}

cudaError_t launch_pose_msg(int model, int64_t N, double tag_z, const double *tagz, const double *x_pred,
                            const double *P_pred_full, double *pose13, double *cov36, cudaStream_t s) {
    if (N <= 0) return cudaSuccess;
    pose_msg_kernel<<<(unsigned)((N + 127) / 128), 128, 0, s>>>(model, N, tag_z, tagz, x_pred, P_pred_full, pose13, cov36);
    return cudaGetLastError();
}

__global__ void fill_kernel(double *p, int64_t n, double v) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) p[i] = v;
}
cudaError_t launch_fill(double *p, int64_t n, double v, cudaStream_t s) {
    if (n <= 0) return cudaSuccess;
    fill_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(p, n, v);
    return cudaGetLastError();
}

// out[i] = sum over r of src[r * n + i] (the rank fold of kfpos_error_hist_allreduce; integers: exact in any order)
__global__ void sum_ranks_u64_kernel(int n_ranks, int64_t n, const unsigned long long *src, unsigned long long *out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    unsigned long long a = 0;
    for (int r = 0; r < n_ranks; ++r) a += src[(int64_t)r * n + i];
    out[i] = a;
}
cudaError_t launch_sum_ranks_u64(int n_ranks, int64_t n, const unsigned long long *src, unsigned long long *out,
                                 cudaStream_t s) {
    if (n <= 0) return cudaSuccess;
    sum_ranks_u64_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(n_ranks, n, src, out);
    return cudaGetLastError();
}

// the fast elementary functions of kfpos_math.cuh evaluated on caller data (accuracy self-test)
__global__ void selftest_math_kernel(int64_t n, const double *x, double *rcp, double *rsq, double *sn, double *cs) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const double v = x[i];
    if (rcp) rcp[i] = fast_rcp(v);
    if (rsq) rsq[i] = fast_rsqrt(v);
    if (sn || cs) {
        double s_, c_;
        fast_sincos(v, &s_, &c_);
        if (sn) sn[i] = s_;
        if (cs) cs[i] = c_;
    }
}

cudaError_t launch_selftest_math(int64_t n, const double *x, double *rcp, double *rsq, double *sn, double *cs,
                                 cudaStream_t s) {
    if (n <= 0) return cudaSuccess;
    selftest_math_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(n, x, rcp, rsq, sn, cs);
    return cudaGetLastError();
}

} // namespace kfpos
