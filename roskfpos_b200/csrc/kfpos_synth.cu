// kfpos_synth.cu -- Monte Carlo input generators, on the device.
//
// synth_k8_kernel: KalmanFilter (K8) batches (BASELINE configs 3 and 5, SURVEY.md §8d): the multi-sensor
// event stream of N independent tags is synthesised on the device, chunk by chunk, straight into the SoA
// tensors the replay kernel streams -- a 64 M-filter x 1000-step run never has its inputs resident (they
// would be 280 GB), only the chunk in flight.
// synth_toa_kernel: ranging epochs for every consumer of a [T][M][N] millimetre range log (T6 / K8 / T9
// ranging replays, the ML batch), with optional missing rangings and exponential NLOS biases (DESIGN §4.5c), and
// optional boxes in the room that bias or remove the rangings whose direct path crosses them (DESIGN §4.5f).
//
// Every value is a pure function of (seed, global filter index, event index, sample index) through
// the counter-based Philox4x32-10 generator (Salmon et al., SC'11; kfpos_synth.cuh), so a filter's stream
// does not depend on how the batch is sharded over GPUs or cut into chunks.
//
// Truth: the planar Lissajous of roskfpos_b200/synth.py  x = 5 + 3 sin(0.20 t + a), y = 5 + 3 sin(0.31 t + b),
// heading th0 + 0.05 t;  a, b, th0 drawn per filter.  K8 samples per 0.1 s macro-step (same schedule as
// synth.MACRO_IMU_MAG / MACRO_FULL): body-frame accelerometer + gyro (IMU), compass, PX4Flow integrals
// (full only), and one epoch of rangings quantised to millimetres.
#include "kfpos_kernels.cuh"
#include "kfpos_synth.cuh"

namespace kfpos {

__global__ void __launch_bounds__(128) synth_k8_kernel(const SynthK8Params p) {
    const int64_t f = (int64_t)blockIdx.x * 128 + threadIdx.x;
    if (f >= p.N) return;
    const int64_t N = p.N;
    const uint64_t gf = (uint64_t)(p.filter0 + f);
    double pa, pb, th0;
    filter_constants(p.seed, gf, pa, pb, th0);
    const double om = 0.05;
    if (p.x0) { // state at t = 0
        const Kin k = kin_at(0.0, pa, pb, th0);
        p.x0[0 * N + f] = k.px; p.x0[1 * N + f] = k.py; p.x0[2 * N + f] = k.vx; p.x0[3 * N + f] = k.vy;
        p.x0[4 * N + f] = 0.0; p.x0[5 * N + f] = 0.0; p.x0[6 * N + f] = k.th; p.x0[7 * N + f] = om;
    }
    for (int e = 0; e < p.n_events; ++e) {
        const SynthEvent ev = p.events[e];
        const Kin k = kin_at(ev.t, pa, pb, th0);
        double sn, cs, n0, n1, n2, n3;
        sincos(k.th, &sn, &cs);
        const uint32_t ge = (uint32_t)ev.global_index;
        switch (ev.kind) {
        case EV_TOA: {
            for (int a = 0; a < p.M; a += 2) {
                normal2(p.seed, gf, ge, (uint32_t)(a >> 1), n0, n1);
                for (int q = 0; q < 2 && a + q < p.M; ++q) {
                    const double ex = k.px - p.anchors.x[a + q], ey = k.py - p.anchors.y[a + q],
                                 ez = p.tag_z - p.anchors.z[a + q];
                    const double d = sqrt(ex * ex + ey * ey + ez * ez) + p.sigma_r * (q ? n1 : n0);
                    const double mm = floor(d * 1000.0);
                    p.ranges[(ev.offset + a + q) * N + f] = mm > 0 ? (int32_t)mm : 0;
                }
            }
            break;
        }
        case EV_IMU: { // gyro z, body-frame accelerations (KF.cpp:573-581)
            normal2(p.seed, gf, ge, 0u, n0, n1);
            normal2(p.seed, gf, ge, 1u, n2, n3);
            p.sensors[(ev.offset + 0) * N + f] = om + 0.29832867780352595 * n0; // sqrt(0.089)
            p.sensors[(ev.offset + 1) * N + f] = cs * k.ax + sn * k.ay + 0.05477225575051661 * n1; // sqrt(0.003)
            p.sensors[(ev.offset + 2) * N + f] = -sn * k.ax + cs * k.ay + 0.05477225575051661 * n2;
            break;
        }
        case EV_PX4: { // integrated flow over 33.333 ms at sensor height 5 m (KF.cpp:100-121)
            normal2(p.seed, gf, ge, 0u, n0, n1);
            const double Tint = 33333.0 / 1e6, H = 5.0;
            p.sensors[(ev.offset + 0) * N + f] = (cs * k.vx + sn * k.vy) * Tint / H + 2e-4 * n0;
            p.sensors[(ev.offset + 1) * N + f] = (-sn * k.vx + cs * k.vy) * Tint / H + 2e-4 * n1;
            p.sensors[(ev.offset + 2) * N + f] = om * Tint;
            p.sensors[(ev.offset + 3) * N + f] = 33333.0;
            p.sensors[(ev.offset + 4) * N + f] = 200.0;
            break;
        }
        default: { // compass: heading + N(0, 0.01^2), wrapped to (-pi, pi]
            normal2(p.seed, gf, ge, 0u, n0, n1);
            const double a = k.th + 0.01 * n0;
            p.sensors[ev.offset * N + f] = a - TWO_PI * floor((a + 0.5 * TWO_PI) / TWO_PI);
            break;
        }
        }
    }
    if (p.truth_end) {
        const Kin k = kin_at(p.t_end, pa, pb, th0);
        p.truth_end[0 * N + f] = k.px; p.truth_end[1 * N + f] = k.py; p.truth_end[2 * N + f] = p.tag_z;
    }
}

cudaError_t launch_synth_k8(const SynthK8Params &p, cudaStream_t s) {
    if (p.N <= 0) return cudaSuccess;
    synth_k8_kernel<<<(unsigned)((p.N + 127) / 128), 128, 0, s>>>(p);
    return cudaGetLastError();
}

// the truth of the filters of BOTH generators, synth_k8_kernel and synth_toa_kernel, at the given times (the
// per-epoch statistics of a chunked run): they share filter_constants and kin_at
__global__ void __launch_bounds__(128) synth_k8_truth_kernel(const SynthTruthParams p) {
    const int64_t f = (int64_t)blockIdx.x * 128 + threadIdx.x;
    if (f >= p.N) return;
    const int64_t N = p.N;
    double pa, pb, th0;
    filter_constants(p.seed, (uint64_t)(p.filter0 + f), pa, pb, th0);
    for (int i = 0; i < p.n_times; ++i) {
        const Kin k = kin_at(p.t[i], pa, pb, th0);
        double *o = p.truth + (int64_t)i * 3 * N + f;
        o[0] = k.px; o[N] = k.py; o[2 * N] = p.tag_z;
    }
}

cudaError_t launch_synth_k8_truth(const SynthTruthParams &p, cudaStream_t s) {
    if (p.N <= 0 || p.n_times <= 0) return cudaSuccess;
    synth_k8_truth_kernel<<<(unsigned)((p.N + 127) / 128), 128, 0, s>>>(p);
    return cudaGetLastError();
}

// Ranging epochs k = 0..n_epochs of global epoch index g = epoch0 + k at time t[k], one thread per filter:
//   d_a = |(x, y, tag_z) - anchor_a| on the truth of filter_constants / kin_at;
//   n_a = component a & 1 of normal2(seed, gf, g, a >> 1);
//   IMPAIR: (u, v) = uniform2(Philox(gf, g, 0x80000000 | a)): missing when u < p_missing, NLOS bias
//           -nlos_mean log(v / p_nlos) when v < p_nlos (v / p_nlos is uniform then: one draw gives both);
//   mm = floor((d_a + sigma_r n_a + bias) * 1000), 0 ("no ranging", TOA.cpp:50) when missing or <= 0.
// MASK: also the NLOS truth, SoA [k][N] uint32 with bit a set when ranging a drew a bias and was written (> 0),
// gathered in a register and stored once per epoch (kfpos_synth_toa_ranges_nlos).
// GEO: the boxes of kfpos_synth_toa_ranges_geo (DESIGN §4.5f).  The slab test of the segment truth -> anchor uses
// only single IEEE operations (no contraction), so a host reproduces every decision from the device truth; the
// Philox draw (gf, g, 0x40000000 | a) of the loss and the exponential bias is made for blocked rangings only.
// The epoch times and the anchors are read from the parameter block: every lane reads the same one at the
// same time (constant-bank broadcast).  Stores: SoA [k][a][N], filter index fastest -- coalesced.
template <typename Out, bool IMPAIR, bool MASK = false, bool GEO = false>
__global__ void __launch_bounds__(128) synth_toa_kernel(const SynthToaParams p) {
    const int64_t f = (int64_t)blockIdx.x * 128 + threadIdx.x;
    if (f >= p.N) return;
    const int64_t N = p.N;
    const uint64_t gf = (uint64_t)(p.filter0 + f);
    double pa, pb, th0;
    filter_constants(p.seed, gf, pa, pb, th0);
    Out *out = (Out *)p.ranges + f;
    const double lim = sizeof(Out) == 2 ? 65535.0 : 2147483647.0;
    for (int k = 0; k < p.n_epochs; ++k) {
        const Kin kn = kin_at(p.t[k], pa, pb, th0);
        const uint32_t g = p.epoch0 + (uint32_t)k;
        uint32_t bits = 0u;
        for (int a = 0; a < p.M; a += 2) {
            double n0, n1;
            normal2(p.seed, gf, g, (uint32_t)(a >> 1), n0, n1);
            for (int q = 0; q < 2 && a + q < p.M; ++q) {
                const int i = a + q;
                const double ex = kn.px - p.anchors.x[i], ey = kn.py - p.anchors.y[i], ez = p.tag_z - p.anchors.z[i];
                const double d = sqrt(ex * ex + ey * ey + ez * ez);
                double r = d + p.sigma_r * (q ? n1 : n0);
                bool missing = false, biased = false;
                if (IMPAIR) {
                    double u, v;
                    uniform2(philox4x32_10((uint32_t)gf, (uint32_t)(gf >> 32), g, 0x80000000u | (uint32_t)i,
                                           (uint32_t)p.seed, (uint32_t)(p.seed >> 32)), u, v);
                    missing = u < p.p_missing;
                    biased = v < p.p_nlos;
                    if (biased) r += -p.nlos_mean * log(v / p.p_nlos);
                }
                if (GEO) {
                    const double tp[3] = {kn.px, kn.py, p.tag_z};
                    const double dv[3] = {__dsub_rn(p.anchors.x[i], kn.px), __dsub_rn(p.anchors.y[i], kn.py),
                                          __dsub_rn(p.anchors.z[i], p.tag_z)};
                    double inv[3];
#pragma unroll
                    for (int j = 0; j < 3; ++j) inv[j] = __ddiv_rn(1.0, dv[j]);
                    bool blocked = false;
                    double excess = 0.0, spread = 0.0, keep = 1.0;
                    for (int o = 0; o < p.n_obstacles; ++o) {
                        const SynthObstacle &b = p.obstacles[o];
                        double enter = 0.0, exit = 1.0;
                        bool inside = true; // every axis with dv == 0 has the truth strictly between the faces
#pragma unroll
                        for (int j = 0; j < 3; ++j) {
                            if (dv[j] != 0.0) {
                                const double s1 = __dmul_rn(__dsub_rn(b.lo[j], tp[j]), inv[j]);
                                const double s2 = __dmul_rn(__dsub_rn(b.hi[j], tp[j]), inv[j]);
                                enter = fmax(enter, fmin(s1, s2));
                                exit = fmin(exit, fmax(s1, s2));
                            } else {
                                inside = inside && b.lo[j] < tp[j] && tp[j] < b.hi[j];
                            }
                        }
                        if (inside && enter < exit) {
                            blocked = true;
                            excess += b.excess_per_m * ((exit - enter) * d);
                            spread += b.spread;
                            keep *= 1.0 - b.p_loss;
                        }
                    }
                    if (blocked) {
                        double u, v;
                        uniform2(philox4x32_10((uint32_t)gf, (uint32_t)(gf >> 32), g, 0x40000000u | (uint32_t)i,
                                               (uint32_t)p.seed, (uint32_t)(p.seed >> 32)), u, v);
                        r += excess;
                        missing = missing || u < 1.0 - keep;
                        if (spread > 0.0) r += -spread * log(v);
                        biased = true;
                    }
                }
                const double mm = floor(r * 1000.0);
                const bool absent = missing || !(mm > 0);
                out[((int64_t)k * p.M + i) * N] = absent ? (Out)0 : (Out)fmin(mm, lim);
                if (MASK && biased && !absent) bits |= 1u << i;
            }
        }
        if (MASK) p.nlos[(int64_t)k * N + f] = bits;
    }
}

template <typename Out, bool MASK, bool GEO>
static void launch_synth_toa_k(const SynthToaParams &p, bool imp, unsigned grid, cudaStream_t s) {
    if (imp) synth_toa_kernel<Out, true, MASK, GEO><<<grid, 128, 0, s>>>(p);
    else synth_toa_kernel<Out, false, MASK, GEO><<<grid, 128, 0, s>>>(p);
}

template <typename Out, bool GEO>
static void launch_synth_toa_m(const SynthToaParams &p, bool imp, unsigned grid, cudaStream_t s) {
    if (p.nlos) launch_synth_toa_k<Out, true, GEO>(p, imp, grid, s);
    else launch_synth_toa_k<Out, false, GEO>(p, imp, grid, s);
}

cudaError_t launch_synth_toa(const SynthToaParams &p, bool u16, cudaStream_t s) {
    if (p.N <= 0 || p.n_epochs <= 0) return cudaSuccess;
    const bool imp = p.p_missing > 0 || p.p_nlos > 0;
    const unsigned grid = (unsigned)((p.N + 127) / 128);
    if (u16) {
        if (p.n_obstacles > 0) launch_synth_toa_m<uint16_t, true>(p, imp, grid, s);
        else launch_synth_toa_m<uint16_t, false>(p, imp, grid, s);
    } else {
        if (p.n_obstacles > 0) launch_synth_toa_m<int32_t, true>(p, imp, grid, s);
        else launch_synth_toa_m<int32_t, false>(p, imp, grid, s);
    }
    return cudaGetLastError();
}

} // namespace kfpos
