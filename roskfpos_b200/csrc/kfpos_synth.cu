// kfpos_synth.cu -- Monte Carlo input generator for KalmanFilter (K8) batches (BASELINE configs 3 and
// 5, SURVEY.md §8d): the multi-sensor event stream of N independent tags is synthesised on the device,
// chunk by chunk, straight into the SoA tensors the replay kernel streams -- a 64 M-filter x 1000-step
// run never has its inputs resident (they would be 280 GB), only the chunk in flight.
//
// Every value is a pure function of (seed, global filter index, event index, sample index) through
// the counter-based Philox4x32-10 generator (Salmon et al., SC'11), so a filter's stream does not
// depend on how the batch is sharded over GPUs or cut into chunks.
//
// Truth: the planar Lissajous of roskfpos_b200/synth.py  x = 5 + 3 sin(0.20 t + a), y = 5 + 3 sin(0.31 t + b),
// heading th0 + 0.05 t;  a, b, th0 drawn per filter.  Samples per 0.1 s macro-step (same schedule as
// synth.MACRO_IMU_MAG / MACRO_FULL): body-frame accelerometer + gyro (IMU), compass, PX4Flow integrals
// (full only), and one epoch of rangings quantised to millimetres.
#include "kfpos_kernels.cuh"

namespace kfpos {

struct Philox {
    uint32_t c[4];
};
KF_DEV Philox philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
        const uint32_t n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
        c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    return Philox{{c0, c1, c2, c3}};
}
// two uniforms in (0, 1) from 4 x 32 bits (53-bit mantissas, never 0)
KF_DEV void uniform2(const Philox &p, double &u0, double &u1) {
    const unsigned long long a = ((unsigned long long)p.c[0] << 32) | p.c[1], b = ((unsigned long long)p.c[2] << 32) | p.c[3];
    u0 = ((double)(a >> 11) + 0.5) * (1.0 / 9007199254740992.0);
    u1 = ((double)(b >> 11) + 0.5) * (1.0 / 9007199254740992.0);
}
// two standard normals (Box-Muller)
KF_DEV void normal2(uint64_t seed, uint64_t filter, uint32_t event, uint32_t sample, double &n0, double &n1) {
    const Philox p = philox4x32_10((uint32_t)filter, (uint32_t)(filter >> 32), event, sample, (uint32_t)seed,
                                   (uint32_t)(seed >> 32));
    double u0, u1, s, c;
    uniform2(p, u0, u1);
    const double rad = sqrt(-2.0 * log(u0));
    sincospi(2.0 * u1, &s, &c);
    n0 = rad * c;
    n1 = rad * s;
}

struct Kin {
    double px, py, vx, vy, ax, ay, th;
};
KF_DEV Kin kin_at(double t, double pa, double pb, double th0) {
    Kin k;
    double s, c;
    sincos(0.20 * t + pa, &s, &c);
    k.px = 5 + 3 * s; k.vx = 0.6 * c; k.ax = -0.12 * s;
    sincos(0.31 * t + pb, &s, &c);
    k.py = 5 + 3 * s; k.vy = 0.93 * c; k.ay = -0.2883 * s;
    k.th = th0 + 0.05 * t;
    return k;
}

constexpr double TWO_PI = 6.283185307179586476925286766559;

// per-filter constants of the truth trajectory (event index 0xFFFFFFFF is reserved for them): phases and heading
KF_DEV void filter_constants(uint64_t seed, uint64_t gf, double &pa, double &pb, double &th0) {
    double ua, ub, uc, ud;
    const Philox q = philox4x32_10((uint32_t)gf, (uint32_t)(gf >> 32), 0xFFFFFFFFu, 0u, (uint32_t)seed,
                                   (uint32_t)(seed >> 32));
    uniform2(q, ua, ub);
    const Philox q2 = philox4x32_10((uint32_t)gf, (uint32_t)(gf >> 32), 0xFFFFFFFFu, 1u, (uint32_t)seed,
                                    (uint32_t)(seed >> 32));
    uniform2(q2, uc, ud);
    pa = ua * TWO_PI;
    pb = ub * TWO_PI;
    th0 = 0.3 + 0.2 * uc;
}

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

// the truth of synth_k8_kernel's filters at the given times (the per-epoch statistics of a chunked run)
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

} // namespace kfpos
