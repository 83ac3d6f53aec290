// kfpos_crlb.cu -- Cramer-Rao lower bound of the position, per epoch, for the rangings a filter or an ML solve
// had, kept, or would have kept with a perfect NLOS detector (kfpos_batch_crlb, DESIGN §4.5e).
//
// One thread per (filter, row).  The M rangings of its epoch give the present set (present_mask, the replay's
// rule), the NLOS mask or the selection (used_mask, the scorer's decoding of `sel`) narrow it to the set S, and
// the Fisher information J = sum_{a in S} g_a g_a^T / v_a of the true position is accumulated in registers: g_a
// = (p - b_a) / |p - b_a| (the x-y part for dim 2, still over the 3-D distance).  Every load is coalesced along
// the filter index.  tr J^-1 and its x-y part come from an LDL^T of J in a fixed order (as epoch_terms factors the
// covariance).  The four terms of a warp's 32 filters are summed by the 32-leaf tree of epoch_stats_flush and
// left in `partials`; the caller folds them over the warp index.  The order of every addition depends on the
// filter index only, so chunking rows changes nothing and aligned power-of-two shards add up bit for bit.
#include "kfpos_kernels.cuh"

namespace kfpos {

namespace {

constexpr int CRLB_BLOCK = 256;

// the four terms of filter f in row r: {tr J^-1, (J^-1)_xx + (J^-1)_yy, 1, 0}, or {0, 0, 0, 1} without a bound
template <int FMT, int D>
__device__ __forceinline__ void crlb_terms(const CrlbParams &p, int64_t r, int64_t f, double (&v)[CRLB_W]) {
    const int64_t N = p.N;
    const double *tr = p.truth + r * 3 * N + f;
    const double px = __ldg(tr), py = __ldg(tr + N), pz = __ldg(tr + 2 * N);
    const unsigned present = present_mask<FMT>(p.ranges, r * p.M * N + f, p.M, N);
    unsigned set = present;
    if (p.set == CRLB_LOS) set &= ~__ldg(p.nlos + r * N + f);
    else if (p.set == CRLB_USED) set &= used_mask(present, p.sel, r, N, f, p.sel_mode);
    // |S| < D: J is singular, though rounding can leave it a tiny positive pivot
    bool ok = __popc(set) >= D && isfinite(px) && isfinite(py) && isfinite(pz);
    const double *var = p.var ? p.var + r * p.M * N + f : nullptr;
    double j00 = 0.0, j10 = 0.0, j11 = 0.0, j20 = 0.0, j21 = 0.0, j22 = 0.0;
#pragma unroll 4
    for (int a = 0; a < p.M; ++a) {
        const bool in = (set >> a) & 1u;
        double w = p.w_scalar;
        if (var) {
            const double va = __ldg(var + (int64_t)a * N);
            ok = ok && (!in || (va > 0.0 && va < INFINITY)); // false for NaN
            w = 1.0 / va;
        }
        const double dx = px - p.anchors.x[a], dy = py - p.anchors.y[a], dz = pz - p.anchors.z[a];
        // a ranging outside S gets g = 0 exactly (and so adds +0), whatever its variance
        const double inv = fast_rsqrt_masked(dx * dx + dy * dy + dz * dz, in);
        const double gx = dx * inv, gy = dy * inv;
        const double wx = in ? w * gx : 0.0, wy = in ? w * gy : 0.0;
        j00 += wx * gx;
        j10 += wy * gx;
        j11 += wy * gy;
        if (D == 3) {
            const double gz = dz * inv, wz = in ? w * gz : 0.0;
            j20 += wz * gx;
            j21 += wz * gy;
            j22 += wz * gz;
        }
    }
    // J = L diag(d) L^T; (J^-1)_ii = sum_k (L^-1)_ki^2 / d_k
    const double d0 = j00;
    const double l10 = j10 / d0;
    const double d1 = j11 - l10 * j10;
    bool pd = d0 > 0.0 && d0 < INFINITY && d1 > 0.0 && d1 < INFINITY;
    const double i0 = 1.0 / d0, i1 = 1.0 / d1;
    double xx = i0 + l10 * l10 * i1, yy = i1, zz = 0.0;
    if (D == 3) {
        const double l20 = j20 / d0;
        const double c = j21 - l20 * j10;
        const double l21 = c / d1;
        const double d2 = j22 - l20 * j20 - l21 * c;
        pd = pd && d2 > 0.0 && d2 < INFINITY;
        const double i2 = 1.0 / d2;
        const double m20 = l20 - l10 * l21; // -(L^-1)_20
        xx += m20 * m20 * i2;
        yy += l21 * l21 * i2;
        zz = i2;
    }
    const double xy = xx + yy;
    const double trace = xy + zz;
    ok = ok && pd && isfinite(trace);
    v[0] = ok ? trace : 0.0;
    v[1] = ok ? xy : 0.0;
    v[2] = ok ? 1.0 : 0.0;
    v[3] = ok ? 0.0 : 1.0;
}

template <int FMT, int D>
__global__ void __launch_bounds__(CRLB_BLOCK) crlb_kernel(const CrlbParams p) {
    const int64_t f = (int64_t)blockIdx.x * CRLB_BLOCK + threadIdx.x;
    if ((f >> 5) >= p.n_warps) return; // whole warps past the batch
    for (int64_t r = blockIdx.y; r < p.n_rows; r += gridDim.y) {
        // lanes without a filter add zeros: the tree of epoch_stats_flush over the warp's filters
        double v[CRLB_W] = {0.0, 0.0, 0.0, 0.0};
        if (f < p.N) crlb_terms<FMT, D>(p, r, f, v);
        epoch_stats_flush<CRLB_W>(Col{v, 1}, 0xffffffffu, p.partials + (r * p.n_warps + (f >> 5)) * CRLB_W);
    }
}

template <int D>
void launch_dim(const CrlbParams &p, dim3 grid, cudaStream_t s) {
    switch (p.fmt) {
    case 0: crlb_kernel<0, D><<<grid, CRLB_BLOCK, 0, s>>>(p); break;
    case 1: crlb_kernel<1, D><<<grid, CRLB_BLOCK, 0, s>>>(p); break;
    default: crlb_kernel<2, D><<<grid, CRLB_BLOCK, 0, s>>>(p); break;
    }
}

} // namespace

cudaError_t launch_crlb(const CrlbParams &p, cudaStream_t s) {
    if (p.N <= 0 || p.n_rows <= 0) return cudaSuccess;
    // filters along x, the fastest block index: the blocks resident at one time read neighbouring parts of a row
    const dim3 grid((unsigned)((p.N + CRLB_BLOCK - 1) / CRLB_BLOCK), (unsigned)(p.n_rows < 65535 ? p.n_rows : 65535));
    if (p.dim == 2) launch_dim<2>(p, grid, s);
    else launch_dim<3>(p, grid, s);
    return cudaGetLastError();
}

} // namespace kfpos
