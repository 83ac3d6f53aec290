// kfpos_synth.cuh -- the counter-based random numbers and the truth kinematics of the Monte Carlo input
// generators (kfpos_synth.cu: synth_k8_kernel, synth_k8_truth_kernel, synth_toa_kernel and synth_walk_kernel).
//
// Every value is a pure function of (seed, global filter index, event index, sample index) through the
// counter-based Philox4x32-10 generator (Salmon et al., SC'11): counter (filter lo, filter hi, event,
// sample), key (seed lo, seed hi).  Event index 0xFFFFFFFF is reserved for the per-filter constants: samples 0
// and 1 for filter_constants, 2 and 3 for the initial position of the random walk (synth_walk_kernel).  Samples
// of an epoch: 0..15 the ranging noise, 0x80000000 | a and 0x40000000 | a its impairments, 0x20000000 and
// 0x20000001 the walk's accelerations -- the walk and the rangings may share one seed without sharing a draw.
#pragma once
#include "kfpos_math.cuh"

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

} // namespace kfpos
