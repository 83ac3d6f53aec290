// kfpos_api.cu -- the C ABI of include/kfpos_b200.h: handle lifetime, host/device
// pointer handling, staging, and dispatch to the kernels.  No torch types, no
// CPU fallback: every path ends in a kernel launch or an error code.
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <new>
#include <vector>

#include "../../include/kfpos_b200.h"
#include <dlfcn.h>

#include "kfpos_kernels.cuh"

using namespace kfpos;

#define CK(call)                                        \
    do {                                                \
        cudaError_t _e = (call);                        \
        if (_e != cudaSuccess) return map_cuda_err(_e); \
    } while (0)

static int map_cuda_err(cudaError_t e) {
    if (e == cudaErrorMemoryAllocation) return KFPOS_ERR_NOMEM;
    return KFPOS_ERR_CUDA;
}

namespace {

struct DevBuf {
    void *p = nullptr;
    size_t cap = 0;
    cudaError_t reserve(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
        cudaError_t e = cudaMalloc(&p, bytes);
        if (e == cudaSuccess) cap = bytes;
        return e;
    }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
    }
};

constexpr int N_SCRATCH = 8;

} // namespace

struct kfpos_batch {
    int device = 0;
    int model = 0;
    int64_t N = 0;
    int n = 0;  // state dimension
    int np = 0; // packed covariance entries
    kfpos_config cfg;
    AnchorTable anchors;
    bool have_anchors = false;
    bool stepped = false; // a measurement has been processed since the (fresh) state was set
    bool imu_seen = false; // T9: an IMU sample has been submitted since set_state (it stays latched)
    double *d_x = nullptr;      // SoA [n][N]
    double *d_P = nullptr;      // SoA [np][N]
    int32_t *d_status = nullptr;
    unsigned long long *d_counters = nullptr;
    double *d_partials = nullptr, *d_out4 = nullptr;
    // ground truth registered with kfpos_batch_set_truth: the replay kernels then leave the error
    // partials of their final state in d_partials (the reduction fused into the last replay step)
    const double *d_truth = nullptr;
    double *d_truth_own = nullptr;
    bool partials_fresh = false;
    bool out4_valid = false; // d_out4 holds the statistics of the current state
    double *d_gather = nullptr; // [n_ranks][4] of kfpos_stats_allreduce
    // per-epoch statistics (kfpos_batch_set_truth_traj): truth rows SoA [es_rows][3][N], per-warp sums
    // [es_rows][n_warps][6] left by the replay kernels, the next output row, and the fold buffers
    const double *d_etruth = nullptr;
    double *d_etruth_own = nullptr, *d_escratch = nullptr, *d_efold = nullptr, *d_eout = nullptr;
    int64_t es_rows = 0, es_cursor = 0, es_fold_rows = 0;
    DevBuf es_gather;
    // K8 / T9 latched sensor samples, SoA rows (see kfpos_k8.cuh)
    double *d_latch = nullptr;
    double *d_latch_u = nullptr; // batch-wide latched IMU covariances
    // ML: straggler queue of the Newton solver (kfpos_mlk.cu)
    void *d_mlq = nullptr;
    int *d_mlq_count = nullptr;
    int mlq_cap = 0;
    int32_t *d_xq = nullptr; // epochs handed to the exact-order solver (kfpos_exact.cu)
    int xq_cap = 0;
    int32_t *d_has = nullptr;
    // ml_initial_position (K8 / T9): while a filter may still be uninitialised the replays run through the
    // general kernel instantiation, which carries the ML-initialisation branch.  Every such launch leaves a
    // flag behind (d_uninit: some filter still has a NaN position); it is copied to pinned host memory behind
    // the launch and looked at -- without waiting -- by the next call.
    bool uninit_possible = false, uninit_pending = false;
    int *d_uninit = nullptr, *h_uninit = nullptr;
    cudaEvent_t ev_uninit = nullptr;
    DevBuf scratch[N_SCRATCH];
    DevBuf stage[2];
    cudaStream_t copy_stream = nullptr;
    cudaEvent_t ev_copied[2] = {nullptr, nullptr}, ev_done[2] = {nullptr, nullptr};
};

namespace {

struct DeviceGuard {
    int prev = -1;
    bool ok = true;
    explicit DeviceGuard(int dev) {
        if (cudaGetDevice(&prev) != cudaSuccess) { ok = false; return; }
        if (prev != dev && cudaSetDevice(dev) != cudaSuccess) ok = false;
    }
    ~DeviceGuard() {
        if (prev >= 0) cudaSetDevice(prev);
    }
};

// true when `p` can be dereferenced by a kernel on this device without staging
bool on_device(const void *p) {
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged;
}

size_t fmt_size(int fmt) { return fmt == KFPOS_FMT_F64_M ? 8 : (fmt == KFPOS_FMT_I32_MM ? 4 : 2); }

// input staging: device pointers pass through, host pointers are copied into
// scratch slot `slot`
int stage_in(kfpos_batch *b, int slot, const void *src, size_t bytes, cudaStream_t s, const void **out) {
    if (!src) { *out = nullptr; return KFPOS_OK; }
    if (on_device(src)) { *out = src; return KFPOS_OK; }
    CK(b->scratch[slot].reserve(bytes));
    CK(cudaMemcpyAsync(b->scratch[slot].p, src, bytes, cudaMemcpyHostToDevice, s));
    *out = b->scratch[slot].p;
    return KFPOS_OK;
}

// output staging: returns the device pointer the kernel should write
int stage_out(kfpos_batch *b, int slot, void *dst, size_t bytes, void **dev, bool *needs_copy) {
    *needs_copy = false;
    if (!dst) { *dev = nullptr; return KFPOS_OK; }
    if (on_device(dst)) { *dev = dst; return KFPOS_OK; }
    CK(b->scratch[slot].reserve(bytes));
    *dev = b->scratch[slot].p;
    *needs_copy = true;
    return KFPOS_OK;
}

int state_dim(int model) {
    switch (model) {
    case KFPOS_MODEL_ML: return 3;
    case KFPOS_MODEL_T6: return 6;
    case KFPOS_MODEL_K8: return 8;
    case KFPOS_MODEL_T9: return 9;
    }
    return 0;
}

RangeStream make_rs(const kfpos_batch *b, const void *ranges, int fmt, double err_scalar, const double *err) {
    RangeStream rs;
    rs.ranges = ranges;
    rs.err = err;
    rs.err_scalar = err_scalar;
    rs.fmt = fmt;
    rs.m_slots = b->anchors.n;
    return rs;
}

int64_t es_warps(const kfpos_batch *b) { return (b->N + 31) / 32; }
// a launch with `rows` output rows: fits the registered truth trajectory (or none is registered)?
int es_check(const kfpos_batch *b, int64_t rows) {
    return (b->d_escratch && b->es_cursor + rows > b->es_rows) ? KFPOS_ERR_INVALID : KFPOS_OK;
}
// the per-epoch statistics pointers of the next launch, then the cursor moves past its `rows` output rows
template <class Params>
void es_bind(kfpos_batch *b, Params &p, int64_t rows) {
    p.n_warps = es_warps(b);
    p.etruth = nullptr;
    p.escratch = nullptr;
    if (!b->d_escratch) return;
    p.etruth = b->d_etruth + b->es_cursor * 3 * b->N;
    p.escratch = b->d_escratch + b->es_cursor * p.n_warps * ES_W;
    b->es_cursor += rows;
}

} // namespace

// ------------------------------------------------------------------------ misc
extern "C" int kfpos_abi_version(void) { return KFPOS_ABI_VERSION; }

extern "C" const char *kfpos_strerror(int code) {
    switch (code) {
    case KFPOS_OK: return "ok";
    case KFPOS_ERR_INVALID: return "invalid argument";
    case KFPOS_ERR_CUDA: return "CUDA error or no CUDA device (this library has no CPU fallback)";
    case KFPOS_ERR_NOMEM: return "out of device memory";
    case KFPOS_ERR_NOT_READY: return "anchors or state not set";
    case KFPOS_ERR_UNSUPPORTED: return "unsupported configuration";
    case KFPOS_ERR_PARSE: return "malformed XML configuration";
    }
    return "unknown error";
}

// -------------------------------------------------------------------- lifetime
extern "C" int kfpos_batch_create(kfpos_batch **out, int device, int model, int64_t n_filters,
                                  const kfpos_config *cfg) {
    if (!out || !cfg || n_filters <= 0 || state_dim(model) == 0) return KFPOS_ERR_INVALID;
    *out = nullptr;
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count <= 0 || device < 0 || device >= count) {
        cudaGetLastError();
        return KFPOS_ERR_CUDA;
    }
    DeviceGuard g(device);
    if (!g.ok) return KFPOS_ERR_CUDA;
    kfpos_batch *b = new (std::nothrow) kfpos_batch();
    if (!b) return KFPOS_ERR_NOMEM;
    b->device = device;
    b->model = model;
    b->N = n_filters;
    b->n = state_dim(model);
    b->np = b->n * (b->n + 1) / 2;
    b->cfg = *cfg;
    memset(&b->anchors, 0, sizeof b->anchors);
    const size_t N = (size_t)n_filters;
    cudaError_t e = cudaSuccess;
    auto alloc = [&](void **p, size_t bytes) {
        if (e == cudaSuccess) e = cudaMalloc(p, bytes);
        if (e == cudaSuccess) e = cudaMemset(*p, 0, bytes);
    };
    alloc((void **)&b->d_counters, CNT_N * sizeof(unsigned long long));
    if (model != KFPOS_MODEL_ML) {
        alloc((void **)&b->d_x, sizeof(double) * b->n * N);
        alloc((void **)&b->d_P, sizeof(double) * b->np * N);
        alloc((void **)&b->d_status, sizeof(int32_t) * N);
        alloc((void **)&b->d_partials, sizeof(double) * 4 * ((N + STATS_CHUNK - 1) / STATS_CHUNK));
        alloc((void **)&b->d_out4, sizeof(double) * 4);
        alloc((void **)&b->d_gather, sizeof(double) * 4 * 1024);
    }
    if (model == KFPOS_MODEL_K8 || model == KFPOS_MODEL_T9) {
        alloc((void **)&b->d_latch, sizeof(double) * 16 * N);
        alloc((void **)&b->d_has, sizeof(int32_t) * N);
        alloc((void **)&b->d_latch_u, sizeof(double) * 32); // [0..15] read by a launch, [16..31] written by it
        alloc((void **)&b->d_uninit, sizeof(int));
        if (e == cudaSuccess) e = cudaHostAlloc((void **)&b->h_uninit, sizeof(int), cudaHostAllocDefault);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&b->ev_uninit, cudaEventDisableTiming);
    }
    if (model == KFPOS_MODEL_ML) {
        if (n_filters > 0x7fffffffLL) {
            kfpos_batch_destroy(b);
            return KFPOS_ERR_UNSUPPORTED;
        }
        b->mlq_cap = (int)(N / 8 + 4096);
        alloc(&b->d_mlq, (size_t)b->mlq_cap * 64 * 2);
        alloc((void **)&b->d_mlq_count, sizeof(int) * 4); // [0..1] straggler queues, [2] exact-order queue
        b->xq_cap = (int)(N / 16 + 1024);
        alloc((void **)&b->d_xq, sizeof(int32_t) * (size_t)b->xq_cap);
    }
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&b->copy_stream, cudaStreamNonBlocking);
    for (int i = 0; i < 2 && e == cudaSuccess; ++i) {
        e = cudaEventCreateWithFlags(&b->ev_copied[i], cudaEventDisableTiming);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&b->ev_done[i], cudaEventDisableTiming);
    }
    if (e != cudaSuccess) {
        kfpos_batch_destroy(b);
        return map_cuda_err(e);
    }
    *out = b;
    return KFPOS_OK;
}

extern "C" void kfpos_batch_destroy(kfpos_batch *b) {
    if (!b) return;
    DeviceGuard g(b->device);
    cudaDeviceSynchronize();
    cudaFree(b->d_x);
    cudaFree(b->d_P);
    cudaFree(b->d_status);
    cudaFree(b->d_counters);
    cudaFree(b->d_partials);
    cudaFree(b->d_out4);
    cudaFree(b->d_truth_own);
    cudaFree(b->d_gather);
    cudaFree(b->d_etruth_own);
    cudaFree(b->d_escratch);
    cudaFree(b->d_efold);
    cudaFree(b->d_eout);
    b->es_gather.release();
    cudaFree(b->d_latch);
    cudaFree(b->d_has);
    cudaFree(b->d_latch_u);
    cudaFree(b->d_uninit);
    if (b->h_uninit) cudaFreeHost(b->h_uninit);
    if (b->ev_uninit) cudaEventDestroy(b->ev_uninit);
    cudaFree(b->d_mlq);
    cudaFree(b->d_mlq_count);
    cudaFree(b->d_xq);
    for (auto &s : b->scratch) s.release();
    for (auto &s : b->stage) s.release();
    for (int i = 0; i < 2; ++i) {
        if (b->ev_copied[i]) cudaEventDestroy(b->ev_copied[i]);
        if (b->ev_done[i]) cudaEventDestroy(b->ev_done[i]);
    }
    if (b->copy_stream) cudaStreamDestroy(b->copy_stream);
    cudaGetLastError();
    delete b;
}

extern "C" int64_t kfpos_batch_size(const kfpos_batch *b) { return b ? b->N : 0; }
extern "C" int kfpos_batch_state_dim(const kfpos_batch *b) { return b ? b->n : 0; }

extern "C" int kfpos_batch_set_anchors(kfpos_batch *b, int n_anchors, const double *xyz) {
    if (!b || !xyz || n_anchors < 0 || n_anchors > KFPOS_MAX_ANCHORS) return KFPOS_ERR_INVALID;
    std::vector<double> host(3 * (size_t)n_anchors);
    if (on_device(xyz)) {
        DeviceGuard g(b->device);
        CK(cudaMemcpy(host.data(), xyz, host.size() * sizeof(double), cudaMemcpyDeviceToHost));
    } else {
        memcpy(host.data(), xyz, host.size() * sizeof(double));
    }
    memset(&b->anchors, 0, sizeof b->anchors);
    for (int i = 0; i < n_anchors; ++i) {
        b->anchors.x[i] = host[3 * i];
        b->anchors.y[i] = host[3 * i + 1];
        b->anchors.z[i] = host[3 * i + 2];
    }
    b->anchors.n = n_anchors;
    b->have_anchors = true;
    return KFPOS_OK;
}

extern "C" int kfpos_batch_set_state(kfpos_batch *b, const double *x, const double *P, void *stream) {
    if (!b || b->model == KFPOS_MODEL_ML || !x) return KFPOS_ERR_INVALID;
    DeviceGuard g(b->device);
    cudaStream_t s = (cudaStream_t)stream;
    const size_t N = (size_t)b->N;
    const bool xd = on_device(x);
    CK(cudaMemcpyAsync(b->d_x, x, sizeof(double) * b->n * N, xd ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, s));
    if (P) {
        const void *pf = nullptr;
        int rc = stage_in(b, 0, P, sizeof(double) * b->n * b->n * N, s, &pf);
        if (rc) return rc;
        CK(launch_pack_cov(b->n, b->N, (const double *)pf, b->d_P, s));
    } else {
        CK(cudaMemsetAsync(b->d_P, 0, sizeof(double) * b->np * N, s));
    }
    CK(cudaMemsetAsync(b->d_status, 0, sizeof(int32_t) * N, s));
    if (b->d_has) CK(cudaMemsetAsync(b->d_has, 0, sizeof(int32_t) * N, s));
    if (b->d_latch) CK(cudaMemsetAsync(b->d_latch, 0, sizeof(double) * 16 * N, s));
    if (b->d_latch_u) CK(cudaMemsetAsync(b->d_latch_u, 0, sizeof(double) * 32, s));
    if (b->model == KFPOS_MODEL_K8) // per-filter tag height (latch row 9): mUWBtagZ = fixedHeight until a 3-D ML init
        CK(launch_fill(b->d_latch + 9 * N, b->N, b->cfg.fixed_height, s));
    b->uninit_possible = b->cfg.ml_initial_position != 0 && (b->model == KFPOS_MODEL_K8 || b->model == KFPOS_MODEL_T9);
    b->uninit_pending = false;
    b->imu_seen = false; // the latches are cleared above
    b->partials_fresh = false;
    b->out4_valid = false;
    b->es_cursor = 0;
    b->stepped = P != nullptr; // a restored checkpoint is a running filter; P0 = 0 is a fresh one
    if (!xd || (P && !on_device(P))) CK(cudaStreamSynchronize(s));
    return KFPOS_OK;
}

extern "C" int kfpos_batch_get_latches(kfpos_batch *b, double *latch, int32_t *has, double *latch_u, void *stream) {
    if (!b || !b->d_latch) return KFPOS_ERR_INVALID;
    DeviceGuard g(b->device);
    cudaStream_t s = (cudaStream_t)stream;
    const size_t N = (size_t)b->N;
    bool sync = false;
    auto out = [&](void *dst, const void *src, size_t bytes) {
        if (!dst) return cudaSuccess;
        const bool d = on_device(dst);
        sync |= !d;
        return cudaMemcpyAsync(dst, src, bytes, d ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost, s);
    };
    CK(out(latch, b->d_latch, sizeof(double) * 16 * N));
    CK(out(has, b->d_has, sizeof(int32_t) * N));
    CK(out(latch_u, b->d_latch_u, sizeof(double) * 16));
    if (sync) CK(cudaStreamSynchronize(s));
    return KFPOS_OK;
}

extern "C" int kfpos_batch_set_latches(kfpos_batch *b, const double *latch, const int32_t *has, const double *latch_u,
                                       void *stream) {
    if (!b || !b->d_latch) return KFPOS_ERR_INVALID;
    DeviceGuard g(b->device);
    cudaStream_t s = (cudaStream_t)stream;
    const size_t N = (size_t)b->N;
    bool sync = false;
    auto in = [&](void *dst, const void *src, size_t bytes) {
        if (!src) return cudaSuccess;
        const bool d = on_device(src);
        sync |= !d;
        return cudaMemcpyAsync(dst, src, bytes, d ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, s);
    };
    CK(in(b->d_latch, latch, sizeof(double) * 16 * N));
    CK(in(b->d_has, has, sizeof(int32_t) * N));
    if (latch_u) {
        CK(in(b->d_latch_u, latch_u, sizeof(double) * 16));
        CK(in(b->d_latch_u + 16, latch_u, sizeof(double) * 16));
    }
    if (has) b->imu_seen = true; // T9: a restored filter may carry a latched IMU sample
    b->stepped = true;
    if (sync) CK(cudaStreamSynchronize(s));
    return KFPOS_OK;
}

extern "C" int kfpos_batch_get_state(kfpos_batch *b, double *x, double *P, int32_t *status, void *stream) {
    if (!b || b->model == KFPOS_MODEL_ML) return KFPOS_ERR_INVALID;
    DeviceGuard g(b->device);
    cudaStream_t s = (cudaStream_t)stream;
    const size_t N = (size_t)b->N;
    bool sync = false;
    if (x) {
        const bool d = on_device(x);
        CK(cudaMemcpyAsync(x, b->d_x, sizeof(double) * b->n * N, d ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost, s));
        sync |= !d;
    }
    if (P) {
        void *dev;
        bool copy;
        const size_t bytes = sizeof(double) * b->n * b->n * N;
        int rc = stage_out(b, 0, P, bytes, &dev, &copy);
        if (rc) return rc;
        CK(launch_unpack_cov(b->n, b->N, b->d_P, (double *)dev, s));
        if (copy) {
            CK(cudaMemcpyAsync(P, dev, bytes, cudaMemcpyDeviceToHost, s));
            sync = true;
        }
    }
    if (status) {
        const bool d = on_device(status);
        CK(cudaMemcpyAsync(status, b->d_status, sizeof(int32_t) * N, d ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost, s));
        sync |= !d;
    }
    if (sync) CK(cudaStreamSynchronize(s));
    return KFPOS_OK;
}

// ------------------------------------------------------------------- TOA steps
namespace {

// launches the model's replay kernel over T steps whose ranges (and optional
// per-ranging errors) are already on the device
int launch_replay(kfpos_batch *b, int T, const double *d_dt, const void *d_ranges, int fmt,
                  double err_scalar, const double *d_err, double *d_traj, int32_t *d_sel, cudaStream_t s,
                  const double *d_dt_f = nullptr);
int run_events(kfpos_batch *b, int n, const kfpos_event *events, const void *d_ranges, int fmt, double err_scalar,
               const double *d_err, const double *d_sensors, double *d_traj, cudaStream_t s,
               const double *d_dt_f = nullptr);

} // namespace

extern "C" int kfpos_batch_replay_toa(kfpos_batch *b, int n_steps, const double *dt, const void *ranges,
                                      int fmt, double err_scalar, const double *err_var, double *traj,
                                      int32_t *sel, void *stream) {
    if (!b || b->model == KFPOS_MODEL_ML || n_steps < 0 || !dt || !ranges) return KFPOS_ERR_INVALID;
    if (fmt < 0 || fmt > 2) return KFPOS_ERR_INVALID;
    if (!b->have_anchors) return KFPOS_ERR_NOT_READY;
    if (n_steps == 0) return KFPOS_OK;
    if (es_check(b, n_steps)) return KFPOS_ERR_INVALID;
    DeviceGuard g(b->device);
    cudaStream_t s = (cudaStream_t)stream;
    const size_t N = (size_t)b->N, M = (size_t)b->anchors.n;
    const int T = n_steps;

    // dt: small, always staged
    CK(b->scratch[1].reserve(sizeof(double) * T));
    CK(cudaMemcpyAsync(b->scratch[1].p, dt, sizeof(double) * T,
                       on_device(dt) ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, s));
    const double *d_dt = (const double *)b->scratch[1].p;

    void *d_traj = nullptr, *d_sel = nullptr;
    bool copy_traj = false, copy_sel = false;
    int rc = stage_out(b, 2, traj, sizeof(double) * 3 * N * T, &d_traj, &copy_traj);
    if (rc) return rc;
    rc = stage_out(b, 3, sel, sizeof(int32_t) * N * T, &d_sel, &copy_sel);
    if (rc) return rc;

    const bool r_dev = on_device(ranges);
    const bool e_dev = !err_var || on_device(err_var);
    if (b->model != KFPOS_MODEL_T6) {
        // K8 / T9: a TOA-only schedule through the event-stream kernel
        std::vector<double> hdt(T);
        if (on_device(dt)) CK(cudaMemcpy(hdt.data(), dt, sizeof(double) * T, cudaMemcpyDeviceToHost));
        else memcpy(hdt.data(), dt, sizeof(double) * T);
        std::vector<kfpos_event> evs(T);
        for (int t = 0; t < T; ++t) {
            memset(&evs[t], 0, sizeof(kfpos_event));
            evs[t].kind = KFPOS_EV_TOA;
            evs[t].dt = hdt[t];
            evs[t].offset = (int64_t)t * (int64_t)M;
        }
        if (sel) return KFPOS_ERR_INVALID; // leave-one-out exists only in T6
        const void *d_r = nullptr, *d_e = nullptr;
        rc = stage_in(b, 4, ranges, M * N * T * fmt_size(fmt), s, &d_r);
        if (rc) return rc;
        rc = stage_in(b, 5, err_var, sizeof(double) * M * N * T, s, &d_e);
        if (rc) return rc;
        rc = run_events(b, T, evs.data(), d_r, fmt, err_scalar, (const double *)d_e, nullptr, (double *)d_traj, s);
        if (rc) return rc;
    } else if (r_dev && e_dev) {
        rc = launch_replay(b, T, d_dt, ranges, fmt, err_scalar, err_var, (double *)d_traj, (int32_t *)d_sel, s);
        if (rc) return rc;
    } else if (!r_dev && err_var == nullptr) {
        // HOST range log: stream it through two device staging buffers, the copy
        // of chunk c+1 overlapping the replay kernel of chunk c.
        // Chunk size: the replay of the LAST chunk is the only kernel time the copies do not hide, so chunks are
        // 1/32 of the log, within [32 MB, 256 MB] (a chunk launch re-reads and re-writes the 192 B of filter state,
        // which bounds how small a chunk is worth making).
        const size_t step_bytes = M * N * fmt_size(fmt);
        size_t chunk_bytes = step_bytes * (size_t)T / 32;
        if (chunk_bytes < ((size_t)32 << 20)) chunk_bytes = (size_t)32 << 20;
        if (chunk_bytes > ((size_t)256 << 20)) chunk_bytes = (size_t)256 << 20;
        size_t chunk_steps = chunk_bytes / (step_bytes ? step_bytes : 1);
        if (chunk_steps < 1) chunk_steps = 1;
        if (chunk_steps > (size_t)T) chunk_steps = (size_t)T;
        for (int i = 0; i < 2; ++i) CK(b->stage[i].reserve(chunk_steps * step_bytes));
        CK(cudaEventRecord(b->ev_done[0], s));
        CK(cudaEventRecord(b->ev_done[1], s));
        int c = 0;
        for (size_t t0 = 0; t0 < (size_t)T; t0 += chunk_steps, ++c) {
            const int k = c & 1;
            const size_t tc = (t0 + chunk_steps <= (size_t)T) ? chunk_steps : (size_t)T - t0;
            CK(cudaStreamWaitEvent(b->copy_stream, b->ev_done[k], 0));
            CK(cudaMemcpyAsync(b->stage[k].p, (const char *)ranges + t0 * step_bytes, tc * step_bytes,
                               cudaMemcpyHostToDevice, b->copy_stream));
            CK(cudaEventRecord(b->ev_copied[k], b->copy_stream));
            CK(cudaStreamWaitEvent(s, b->ev_copied[k], 0));
            rc = launch_replay(b, (int)tc, d_dt + t0, b->stage[k].p, fmt, err_scalar, nullptr,
                               d_traj ? (double *)d_traj + t0 * 3 * N : nullptr,
                               d_sel ? (int32_t *)d_sel + t0 * N : nullptr, s);
            if (rc) return rc;
            CK(cudaEventRecord(b->ev_done[k], s));
        }
    } else {
        // host ranges with per-ranging errors (or mixed): stage both whole
        const void *d_r = nullptr, *d_e = nullptr;
        rc = stage_in(b, 4, ranges, M * N * T * fmt_size(fmt), s, &d_r);
        if (rc) return rc;
        rc = stage_in(b, 5, err_var, sizeof(double) * M * N * T, s, &d_e);
        if (rc) return rc;
        rc = launch_replay(b, T, d_dt, d_r, fmt, err_scalar, (const double *)d_e, (double *)d_traj,
                           (int32_t *)d_sel, s);
        if (rc) return rc;
    }
    if (copy_traj) CK(cudaMemcpyAsync(traj, d_traj, sizeof(double) * 3 * N * T, cudaMemcpyDeviceToHost, s));
    if (copy_sel) CK(cudaMemcpyAsync(sel, d_sel, sizeof(int32_t) * N * T, cudaMemcpyDeviceToHost, s));
    if (copy_traj || copy_sel || !r_dev || !e_dev) CK(cudaStreamSynchronize(s));
    return KFPOS_OK;
}

extern "C" int kfpos_batch_replay_epochs(kfpos_batch *b, int n_steps, const double *dt_per_filter, const void *ranges,
                                         int fmt, double err_scalar, const double *err_var, double *traj,
                                         void *stream) {
    if (!b || n_steps < 0 || !dt_per_filter || !ranges) return KFPOS_ERR_INVALID;
    if (b->model != KFPOS_MODEL_T6 && b->model != KFPOS_MODEL_K8 && b->model != KFPOS_MODEL_T9) return KFPOS_ERR_INVALID;
    if (fmt < 0 || fmt > 2) return KFPOS_ERR_INVALID;
    if (!b->have_anchors) return KFPOS_ERR_NOT_READY;
    if (n_steps == 0) return KFPOS_OK;
    if (es_check(b, n_steps)) return KFPOS_ERR_INVALID;
    DeviceGuard g(b->device);
    cudaStream_t s = (cudaStream_t)stream;
    const size_t N = (size_t)b->N, M = (size_t)b->anchors.n, T = (size_t)n_steps;
    const void *d_dtf = nullptr, *d_r = nullptr, *d_e = nullptr;
    int rc = stage_in(b, 1, dt_per_filter, sizeof(double) * N * T, s, &d_dtf);
    if (rc) return rc;
    if ((rc = stage_in(b, 4, ranges, M * N * T * fmt_size(fmt), s, &d_r))) return rc;
    if ((rc = stage_in(b, 5, err_var, sizeof(double) * M * N * T, s, &d_e))) return rc;
    void *d_traj = nullptr;
    bool copy_traj = false;
    if ((rc = stage_out(b, 2, traj, sizeof(double) * 3 * N * T, &d_traj, &copy_traj))) return rc;
    if (b->model == KFPOS_MODEL_T6) {
        rc = launch_replay(b, n_steps, nullptr, d_r, fmt, err_scalar, (const double *)d_e, (double *)d_traj, nullptr, s,
                           (const double *)d_dtf);
    } else { // K8 / T9: the epochs as a schedule of ranging events whose time steps are per filter
        std::vector<kfpos_event> evs(T);
        for (size_t t = 0; t < T; ++t) {
            memset(&evs[t], 0, sizeof(kfpos_event));
            evs[t].kind = KFPOS_EV_TOA;
            evs[t].offset = (int64_t)t * (int64_t)M;
        }
        rc = run_events(b, n_steps, evs.data(), d_r, fmt, err_scalar, (const double *)d_e, nullptr, (double *)d_traj, s,
                        (const double *)d_dtf);
    }
    if (rc) return rc;
    if (copy_traj) CK(cudaMemcpyAsync(traj, d_traj, sizeof(double) * 3 * N * T, cudaMemcpyDeviceToHost, s));
    if (copy_traj || !on_device(ranges) || !on_device(dt_per_filter) || (err_var && !on_device(err_var)))
        CK(cudaStreamSynchronize(s));
    return KFPOS_OK;
}

extern "C" int kfpos_batch_step_toa(kfpos_batch *b, double dt, const void *ranges, int fmt, double err_scalar,
                                    const double *err_var, void *stream) {
    return kfpos_batch_replay_toa(b, 1, &dt, ranges, fmt, err_scalar, err_var, nullptr, nullptr, stream);
}

namespace {

int launch_replay(kfpos_batch *b, int T, const double *d_dt, const void *d_ranges, int fmt,
                  double err_scalar, const double *d_err, double *d_traj, int32_t *d_sel, cudaStream_t s,
                  const double *d_dt_f) {
    const RangeStream rs = make_rs(b, d_ranges, fmt, err_scalar, d_err);
    b->stepped = true;
    switch (b->model) {
    case KFPOS_MODEL_T6: {
        T6Params p;
        p.anchors = b->anchors;
        p.rs = rs;
        p.N = b->N;
        p.T = T;
        p.ignore_worst = b->cfg.ignore_worst_anchor;
        p.variant = b->cfg.variant;
        p.n_ignore = b->cfg.num_ignored_rangings;
        p.best_mode = b->cfg.best_mode;
        p.ignore_thr = b->cfg.ignore_cost_threshold;
        p.accel_noise = b->cfg.accel_noise;
        p.dt = d_dt;
        p.dt_f = d_dt_f;
        p.x = b->d_x;
        p.P = b->d_P;
        p.status = b->d_status;
        p.traj = d_traj;
        p.sel = d_sel;
        p.counters = b->d_counters;
        p.truth = b->d_truth;
        p.partials = b->d_partials;
        es_bind(b, p, T);
        CK(launch_t6_replay(p, s));
        b->partials_fresh = b->d_truth != nullptr;
        b->out4_valid = false;
        return KFPOS_OK;
    }
    default: return KFPOS_ERR_UNSUPPORTED;
    }
}

} // namespace

// ------------------------------------------------------------ event schedules
namespace {

K8Cfg make_k8cfg(const kfpos_batch *b) {
    K8Cfg c;
    c.accel_noise = b->cfg.accel_noise;
    c.jolt = b->cfg.jolt;
    c.tag_z = b->cfg.fixed_height;
    c.px4_height = b->cfg.px4_sensor_height;
    c.arm1 = b->cfg.px4_arm_p0;
    c.arm2 = b->cfg.px4_arm_p1;
    c.px4_cov_vel = b->cfg.px4_cov_velocity;
    c.px4_cov_gyro = b->cfg.px4_cov_gyro_z;
    c.imu_cov_acc = b->cfg.imu_cov_acc;
    c.imu_cov_gyro = b->cfg.imu_cov_gyro_z;
    c.mag_offset = b->cfg.mag_angle_offset;
    c.mag_cov = b->cfg.mag_cov;
    c.imu_fix_acc = b->cfg.imu_use_fixed_cov_acc;
    c.imu_fix_gyro = b->cfg.imu_use_fixed_cov_gyro_z;
    c.variant = b->cfg.variant;
    c.n_ignore = b->cfg.num_ignored_rangings;
    c.best_mode = b->cfg.best_mode;
    c.zero_tz = b->cfg.ml2d_zero_tentative_z != 0;
    c.use_fixed_height = b->cfg.use_fixed_height != 0;
    // after a 3-D initialisation the tag height is per filter (latch row 9), so the flag stays on in that mode;
    // in 2-D mode it is dropped once a launch has ended with every filter initialised (poll_uninit)
    c.ml_init = b->cfg.ml_initial_position != 0 && (b->uninit_possible || !c.use_fixed_height);
    return c;
}

// ml_initial_position: has the previous launch's "some filter is still uninitialised" flag arrived, and is it 0?
void poll_uninit(kfpos_batch *b) {
    if (!b->uninit_possible || !b->uninit_pending) return;
    if (cudaEventQuery(b->ev_uninit) != cudaSuccess) {
        cudaGetLastError();
        return;
    }
    b->uninit_pending = false;
    if (*b->h_uninit == 0) b->uninit_possible = false;
}
int arm_uninit(kfpos_batch *b, cudaStream_t s) {
    CK(cudaMemsetAsync(b->d_uninit, 0, sizeof(int), s));
    return KFPOS_OK;
}
int fetch_uninit(kfpos_batch *b, cudaStream_t s) {
    CK(cudaMemcpyAsync(b->h_uninit, b->d_uninit, sizeof(int), cudaMemcpyDeviceToHost, s));
    CK(cudaEventRecord(b->ev_uninit, s));
    b->uninit_pending = true;
    return KFPOS_OK;
}

// events: HOST array; every data pointer already on the device
int run_events(kfpos_batch *b, int n, const kfpos_event *events, const void *d_ranges, int fmt, double err_scalar,
               const double *d_err, const double *d_sensors, double *d_traj, cudaStream_t s, const double *d_dt_f) {
    static_assert(sizeof(kfpos_event) == sizeof(EventDesc), "kfpos_event and EventDesc must have one layout");
    if (n <= 0) return KFPOS_OK;
    b->stepped = true;
    CK(b->scratch[7].reserve(sizeof(EventDesc) * (size_t)n));
    CK(cudaMemcpyAsync(b->scratch[7].p, events, sizeof(EventDesc) * (size_t)n, cudaMemcpyHostToDevice, s));
    const RangeStream rs = make_rs(b, d_ranges, fmt, err_scalar, d_err);
    poll_uninit(b);
    const bool track_uninit = b->uninit_possible;
    int64_t n_toa = 0;
    for (int i = 0; i < n; ++i) n_toa += events[i].kind == KFPOS_EV_TOA;
    if (track_uninit) {
        int rc = arm_uninit(b, s);
        if (rc) return rc;
    }
    switch (b->model) {
    case KFPOS_MODEL_K8: {
        K8Params p;
        p.anchors = b->anchors;
        p.cfg = make_k8cfg(b);
        p.rs = rs;
        p.sensors = d_sensors;
        p.events = (const EventDesc *)b->scratch[7].p;
        p.n_events = n;
        p.N = b->N;
        p.x = b->d_x;
        p.P = b->d_P;
        p.status = b->d_status;
        p.latch = b->d_latch;
        p.has = b->d_has;
        p.latch_u = b->d_latch_u;
        p.uninit = track_uninit ? b->d_uninit : nullptr;
        p.dt_f = d_dt_f;
        p.traj = d_traj;
        p.counters = b->d_counters;
        p.truth = b->d_truth;
        p.partials = b->d_partials;
        es_bind(b, p, n_toa);
        CK(launch_k8_replay(p, s));
        CK(cudaMemcpyAsync(b->d_latch_u, b->d_latch_u + 16, sizeof(double) * 16, cudaMemcpyDeviceToDevice, s));
        b->partials_fresh = b->d_truth != nullptr;
        b->out4_valid = false;
        break;
    }
    case KFPOS_MODEL_T9: {
        T9Params p;
        p.anchors = b->anchors;
        p.accel_noise = b->cfg.accel_noise;
        p.jolt = b->cfg.jolt;
        p.rs = rs;
        p.sensors = d_sensors;
        p.events = (const EventDesc *)b->scratch[7].p;
        p.n_events = n;
        p.N = b->N;
        p.x = b->d_x;
        p.P = b->d_P;
        p.status = b->d_status;
        p.latch = b->d_latch;
        p.has = b->d_has;
        p.latch_u = b->d_latch_u;
        for (int i = 0; i < n; ++i) b->imu_seen = b->imu_seen || events[i].kind == KFPOS_EV_IMU;
        p.no_imu = b->imu_seen ? 0 : 1;
        p.variant = b->cfg.variant;
        p.n_ignore = b->cfg.num_ignored_rangings;
        p.best_mode = b->cfg.best_mode;
        p.ml_init = track_uninit ? 1 : 0;
        p.uninit = track_uninit ? b->d_uninit : nullptr;
        p.dt_f = d_dt_f;
        p.traj = d_traj;
        p.counters = b->d_counters;
        p.truth = b->d_truth;
        p.partials = b->d_partials;
        es_bind(b, p, n_toa);
        CK(launch_t9_replay(p, s));
        CK(cudaMemcpyAsync(b->d_latch_u, b->d_latch_u + 16, sizeof(double) * 16, cudaMemcpyDeviceToDevice, s));
        b->partials_fresh = b->d_truth != nullptr;
        b->out4_valid = false;
        break;
    }
    default: return KFPOS_ERR_INVALID;
    }
    if (track_uninit) {
        int rc = fetch_uninit(b, s);
        if (rc) return rc;
    }
    // (the host event array may be a temporary of the caller: a copy from pageable memory has left the
    // caller's buffer when cudaMemcpyAsync returns, so no synchronisation is needed here)
    return KFPOS_OK;
}

} // namespace

static int replay_events_impl(kfpos_batch *b, int n_events, const kfpos_event *events, const double *dt_per_filter,
                              const void *ranges, int fmt, double err_scalar, const double *err_var,
                              const double *sensors, int64_t sensor_rows, double *traj, void *stream) {
    if (!b || (b->model != KFPOS_MODEL_K8 && b->model != KFPOS_MODEL_T9) || n_events < 0 || !events)
        return KFPOS_ERR_INVALID;
    if (fmt < 0 || fmt > 2) return KFPOS_ERR_INVALID;
    if (!b->have_anchors) return KFPOS_ERR_NOT_READY;
    if (n_events == 0) return KFPOS_OK;
    DeviceGuard g(b->device);
    cudaStream_t s = (cudaStream_t)stream;
    const size_t N = (size_t)b->N, M = (size_t)b->anchors.n;
    int64_t range_rows = 0, n_toa = 0;
    for (int e = 0; e < n_events; ++e) {
        const kfpos_event &ev = events[e];
        if (ev.kind < KFPOS_EV_TOA || ev.kind > KFPOS_EV_COMPASS || ev.offset < 0) return KFPOS_ERR_INVALID;
        if (b->model == KFPOS_MODEL_T9 && ev.kind != KFPOS_EV_TOA && ev.kind != KFPOS_EV_IMU) return KFPOS_ERR_INVALID;
        if (ev.kind == KFPOS_EV_TOA) {
            if (!ranges) return KFPOS_ERR_INVALID;
            if (ev.offset + (int64_t)M > range_rows) range_rows = ev.offset + (int64_t)M;
            ++n_toa;
        } else {
            const int rows = ev.kind == KFPOS_EV_PX4 ? 5 : ev.kind == KFPOS_EV_IMU ? 3 : ev.kind == KFPOS_EV_MAG ? 2 : 1;
            if (!sensors || ev.offset + rows > sensor_rows) return KFPOS_ERR_INVALID;
        }
    }
    if (es_check(b, n_toa)) return KFPOS_ERR_INVALID;
    const void *d_r = nullptr, *d_e = nullptr, *d_s = nullptr;
    int rc = stage_in(b, 4, ranges, (size_t)range_rows * N * fmt_size(fmt), s, &d_r);
    if (rc) return rc;
    rc = stage_in(b, 5, err_var, sizeof(double) * (size_t)range_rows * N, s, &d_e);
    if (rc) return rc;
    rc = stage_in(b, 6, sensors, sizeof(double) * (size_t)sensor_rows * N, s, &d_s);
    if (rc) return rc;
    void *d_traj = nullptr;
    bool copy_traj = false;
    rc = stage_out(b, 2, traj, sizeof(double) * 3 * N * (size_t)n_toa, &d_traj, &copy_traj);
    if (rc) return rc;
    const void *d_dtf = nullptr;
    if ((rc = stage_in(b, 1, dt_per_filter, sizeof(double) * N * (size_t)n_events, s, &d_dtf))) return rc;
    rc = run_events(b, n_events, events, d_r, fmt, err_scalar, (const double *)d_e, (const double *)d_s,
                    (double *)d_traj, s, (const double *)d_dtf);
    if (rc) return rc;
    if (copy_traj) {
        CK(cudaMemcpyAsync(traj, d_traj, sizeof(double) * 3 * N * (size_t)n_toa, cudaMemcpyDeviceToHost, s));
        CK(cudaStreamSynchronize(s));
    }
    return KFPOS_OK;
}

extern "C" int kfpos_batch_replay_events(kfpos_batch *b, int n_events, const kfpos_event *events, const void *ranges,
                                         int fmt, double err_scalar, const double *err_var, const double *sensors,
                                         int64_t sensor_rows, double *traj, void *stream) {
    return replay_events_impl(b, n_events, events, nullptr, ranges, fmt, err_scalar, err_var, sensors, sensor_rows, traj,
                              stream);
}

extern "C" int kfpos_batch_replay_events_ragged(kfpos_batch *b, int n_events, const kfpos_event *events,
                                                const double *dt_per_filter, const void *ranges, int fmt,
                                                double err_scalar, const double *err_var, const double *sensors,
                                                int64_t sensor_rows, double *traj, void *stream) {
    if (!dt_per_filter) return KFPOS_ERR_INVALID;
    return replay_events_impl(b, n_events, events, dt_per_filter, ranges, fmt, err_scalar, err_var, sensors, sensor_rows,
                              traj, stream);
}

namespace {

// one non-TOA event whose payload rows are gathered into scratch slot 6
int single_sensor_event(kfpos_batch *b, int kind, double dt, const double *const *rows, int n_rows,
                        const double aux[9], cudaStream_t s) {
    const size_t N = (size_t)b->N;
    CK(b->scratch[6].reserve(sizeof(double) * N * (size_t)n_rows));
    double *dst = (double *)b->scratch[6].p;
    for (int i = 0; i < n_rows; ++i) {
        if (!rows[i]) return KFPOS_ERR_INVALID;
        CK(cudaMemcpyAsync(dst + (size_t)i * N, rows[i], sizeof(double) * N,
                           on_device(rows[i]) ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, s));
    }
    kfpos_event ev;
    memset(&ev, 0, sizeof ev);
    ev.kind = kind;
    ev.dt = dt;
    ev.offset = 0;
    if (aux) memcpy(ev.aux, aux, sizeof ev.aux);
    return run_events(b, 1, &ev, nullptr, KFPOS_FMT_F64_M, 1.0, nullptr, dst, nullptr, s);
}

} // namespace

extern "C" int kfpos_batch_step_px4(kfpos_batch *b, double dt, const double *integration_x,
                                    const double *integration_y, const double *integration_rot_z,
                                    const double *integration_time_us, const int32_t *quality, void *stream) {
    if (!b || b->model != KFPOS_MODEL_K8 || !quality) return KFPOS_ERR_INVALID;
    DeviceGuard g(b->device);
    cudaStream_t s = (cudaStream_t)stream;
    const size_t N = (size_t)b->N;
    const void *d_q = nullptr;
    int rc = stage_in(b, 5, quality, sizeof(int32_t) * N, s, &d_q);
    if (rc) return rc;
    CK(b->scratch[3].reserve(sizeof(double) * N));
    CK(launch_i32_to_f64(b->N, (const int32_t *)d_q, (double *)b->scratch[3].p, s));
    const double *rows[5] = {integration_x, integration_y, integration_rot_z, integration_time_us,
                             (const double *)b->scratch[3].p};
    return single_sensor_event(b, KFPOS_EV_PX4, dt, rows, 5, nullptr, s);
}

extern "C" int kfpos_batch_step_imu(kfpos_batch *b, double dt, const double *ang_vel, const double *cov_ang_vel,
                                    const double *lin_acc, const double *cov_acc, void *stream) {
    if (!b || (b->model != KFPOS_MODEL_K8 && b->model != KFPOS_MODEL_T9) || !lin_acc) return KFPOS_ERR_INVALID;
    DeviceGuard g(b->device);
    cudaStream_t s = (cudaStream_t)stream;
    const size_t N = (size_t)b->N;
    double aux[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
    if (b->model == KFPOS_MODEL_K8) {
        if (!ang_vel) return KFPOS_ERR_INVALID;
        if (cov_acc) { aux[0] = cov_acc[0]; aux[1] = cov_acc[1]; aux[2] = cov_acc[3]; aux[3] = cov_acc[4]; }
        if (cov_ang_vel) aux[4] = cov_ang_vel[8];
        const double *rows[3] = {ang_vel + 2 * N, lin_acc, lin_acc + N};
        return single_sensor_event(b, KFPOS_EV_IMU, dt, rows, 3, aux, s);
    }
    if (cov_acc) memcpy(aux, cov_acc, sizeof aux);
    const double *rows[3] = {lin_acc, lin_acc + N, lin_acc + 2 * N};
    return single_sensor_event(b, KFPOS_EV_IMU, dt, rows, 3, aux, s);
}

extern "C" int kfpos_batch_step_mag(kfpos_batch *b, double dt, const double *mag, void *stream) {
    if (!b || b->model != KFPOS_MODEL_K8 || !mag) return KFPOS_ERR_INVALID;
    DeviceGuard g(b->device);
    const double *rows[2] = {mag, mag + (size_t)b->N};
    return single_sensor_event(b, KFPOS_EV_MAG, dt, rows, 2, nullptr, (cudaStream_t)stream);
}

extern "C" int kfpos_batch_step_compass(kfpos_batch *b, double dt, const double *compass, void *stream) {
    if (!b || b->model != KFPOS_MODEL_K8 || !compass) return KFPOS_ERR_INVALID;
    DeviceGuard g(b->device);
    const double *rows[1] = {compass};
    return single_sensor_event(b, KFPOS_EV_COMPASS, dt, rows, 1, nullptr, (cudaStream_t)stream);
}

// --------------------------------------------------------------------- getPose
extern "C" int kfpos_batch_get_pose(kfpos_batch *b, double dt, double *x_pred, double *P_pred, void *stream) {
    if (!b || b->model == KFPOS_MODEL_ML) return KFPOS_ERR_INVALID;
    DeviceGuard g(b->device);
    cudaStream_t s = (cudaStream_t)stream;
    const size_t N = (size_t)b->N;
    void *dx = nullptr, *dP = nullptr;
    bool cx = false, cP = false;
    int rc = stage_out(b, 2, x_pred, sizeof(double) * b->n * N, &dx, &cx);
    if (rc) return rc;
    rc = stage_out(b, 3, P_pred, sizeof(double) * b->n * b->n * N, &dP, &cP);
    if (rc) return rc;
    switch (b->model) {
    case KFPOS_MODEL_T6:
        CK(launch_t6_get_pose(b->N, dt, b->cfg.accel_noise, b->d_x, b->d_P, (double *)dx, (double *)dP, s));
        break;
    case KFPOS_MODEL_K8:
        CK(launch_k8_get_pose(b->N, dt, b->cfg.accel_noise, b->cfg.jolt, b->d_x, b->d_P, (double *)dx, (double *)dP, s));
        break;
    case KFPOS_MODEL_T9:
        CK(launch_t9_get_pose(b->N, dt, b->cfg.jolt, b->d_x, b->d_P, (double *)dx, (double *)dP, s));
        break;
    default: return KFPOS_ERR_UNSUPPORTED;
    }
    if (cx) CK(cudaMemcpyAsync(x_pred, dx, sizeof(double) * b->n * N, cudaMemcpyDeviceToHost, s));
    if (cP) CK(cudaMemcpyAsync(P_pred, dP, sizeof(double) * b->n * b->n * N, cudaMemcpyDeviceToHost, s));
    if (cx || cP) CK(cudaStreamSynchronize(s));
    return KFPOS_OK;
}

extern "C" int kfpos_batch_get_pose_msg(kfpos_batch *b, double dt, double *pose13, double *cov36, void *stream) {
    if (!b || b->model == KFPOS_MODEL_ML) return KFPOS_ERR_INVALID;
    if (!b->stepped) return KFPOS_ERR_NOT_READY; // getPose returns false before the first measurement
    DeviceGuard g(b->device);
    cudaStream_t s = (cudaStream_t)stream;
    const size_t N = (size_t)b->N;
    CK(b->scratch[2].reserve(sizeof(double) * b->n * N));
    CK(b->scratch[3].reserve(sizeof(double) * b->n * b->n * N));
    double *dx = (double *)b->scratch[2].p, *dP = (double *)b->scratch[3].p;
    int rc = kfpos_batch_get_pose(b, dt, dx, dP, stream);
    if (rc) return rc;
    void *d_pose = nullptr, *d_cov = nullptr;
    bool c_pose = false, c_cov = false;
    if ((rc = stage_out(b, 4, pose13, sizeof(double) * 13 * N, &d_pose, &c_pose))) return rc;
    if ((rc = stage_out(b, 5, cov36, sizeof(double) * 36 * N, &d_cov, &c_cov))) return rc;
    const int model = b->model == KFPOS_MODEL_T6 ? 1 : (b->model == KFPOS_MODEL_K8 ? 2 : 3);
    // K8 without useFixedHeight: the tag height of an ML-initialised filter is its own (KF.cpp:256-257, 328-332)
    const double *tagz = (b->model == KFPOS_MODEL_K8 && b->cfg.ml_initial_position && !b->cfg.use_fixed_height)
                             ? b->d_latch + 9 * N : nullptr;
    CK(launch_pose_msg(model, b->N, b->cfg.fixed_height, tagz, dx, dP, (double *)d_pose, (double *)d_cov, s));
    if (c_pose) CK(cudaMemcpyAsync(pose13, d_pose, sizeof(double) * 13 * N, cudaMemcpyDeviceToHost, s));
    if (c_cov) CK(cudaMemcpyAsync(cov36, d_cov, sizeof(double) * 36 * N, cudaMemcpyDeviceToHost, s));
    if (c_pose || c_cov) CK(cudaStreamSynchronize(s));
    return KFPOS_OK;
}

// -------------------------------------------------------------------------- ML
extern "C" int kfpos_batch_ml_solve(kfpos_batch *b, const void *ranges, int fmt, double err_scalar,
                                    const double *err_var, double *pos, double *cov, int32_t *iters,
                                    int32_t *sel, int32_t *status, void *stream) {
    if (!b || b->model != KFPOS_MODEL_ML || !ranges || fmt < 0 || fmt > 2) return KFPOS_ERR_INVALID;
    if (!b->have_anchors) return KFPOS_ERR_NOT_READY;
    DeviceGuard g(b->device);
    cudaStream_t s = (cudaStream_t)stream;
    const size_t N = (size_t)b->N, M = (size_t)b->anchors.n;
    const void *d_r = nullptr, *d_e = nullptr;
    int rc = stage_in(b, 0, ranges, M * N * fmt_size(fmt), s, &d_r);
    if (rc) return rc;
    rc = stage_in(b, 1, err_var, sizeof(double) * M * N, s, &d_e);
    if (rc) return rc;
    void *d_pos, *d_cov, *d_it, *d_sel, *d_st;
    bool c_pos, c_cov, c_it, c_sel, c_st;
    if ((rc = stage_out(b, 2, pos, sizeof(double) * 3 * N, &d_pos, &c_pos))) return rc;
    if ((rc = stage_out(b, 3, cov, sizeof(double) * 9 * N, &d_cov, &c_cov))) return rc;
    if ((rc = stage_out(b, 4, iters, sizeof(int32_t) * N, &d_it, &c_it))) return rc;
    if ((rc = stage_out(b, 5, sel, sizeof(int32_t) * 2 * N, &d_sel, &c_sel))) return rc;
    if ((rc = stage_out(b, 6, status, sizeof(int32_t) * N, &d_st, &c_st))) return rc;
    MlParams p;
    p.anchors = b->anchors;
    p.rs = make_rs(b, d_r, fmt, err_scalar, (const double *)d_e);
    p.N = b->N;
    p.use2d = b->cfg.use2d;
    p.zero_tz = b->cfg.ml2d_zero_tentative_z != 0;
    p._pad = 0;
    p.variant = b->cfg.variant;
    p.n_ignore = b->cfg.num_ignored_rangings;
    p.best_mode = b->cfg.best_mode;
    p.start[0] = b->cfg.ml_start[0];
    p.start[1] = b->cfg.ml_start[1];
    p.start[2] = b->cfg.ml_start[2];
    p.min_z = b->cfg.min_z;
    p.max_z = b->cfg.max_z;
    p.pos = (double *)d_pos;
    p.cov = (double *)d_cov;
    p.iters = (int32_t *)d_it;
    p.sel = (int32_t *)d_sel;
    p.status = (int32_t *)d_st;
    p.counters = b->d_counters;
    p.queue[0] = b->d_mlq;
    p.queue[1] = (char *)b->d_mlq + (size_t)b->mlq_cap * 64;
    p.queue_count = b->d_mlq_count;
    p.queue_cap = b->mlq_cap;
    p.q_in = nullptr; p.q_in_count = nullptr; p.q_out = nullptr; p.q_out_count = nullptr;
    p.first_cap = 10000u;
    p.coop_min = 0; p.coop_max = 0;
    p.exact_mode = b->cfg.ml_exact_order;
    p.xq = b->d_xq;
    p.xq_count = b->d_mlq_count + 2;
    p.xq_cap = b->xq_cap;
    p.xw_scratch = nullptr;
    p.xw_scratch_bytes = 0;
    p.stream_counter = b->d_mlq_count + 3;
    if (p.variant == 2 && !p.use2d && p.exact_mode >= 0) { // parked subset solves of the 3-D BestGroup scan
        const size_t bytes = ml_exact_scratch_bytes(ml_exact_scratch_epochs(b->N));
        CK(b->scratch[7].reserve(bytes));
        p.xw_scratch = b->scratch[7].p;
        p.xw_scratch_bytes = bytes;
    }
    CK(launch_ml_solve(p, s));
    if (c_pos) CK(cudaMemcpyAsync(pos, d_pos, sizeof(double) * 3 * N, cudaMemcpyDeviceToHost, s));
    if (c_cov) CK(cudaMemcpyAsync(cov, d_cov, sizeof(double) * 9 * N, cudaMemcpyDeviceToHost, s));
    if (c_it) CK(cudaMemcpyAsync(iters, d_it, sizeof(int32_t) * N, cudaMemcpyDeviceToHost, s));
    if (c_sel) CK(cudaMemcpyAsync(sel, d_sel, sizeof(int32_t) * 2 * N, cudaMemcpyDeviceToHost, s));
    if (c_st) CK(cudaMemcpyAsync(status, d_st, sizeof(int32_t) * N, cudaMemcpyDeviceToHost, s));
    if (c_pos || c_cov || c_it || c_sel || c_st || !on_device(ranges)) CK(cudaStreamSynchronize(s));
    return KFPOS_OK;
}

// ------------------------------------------------------------ epoch assembler
namespace {
// temporary device copy of a host array (or the device pointer itself)
struct TmpIn {
    const void *d = nullptr;
    void *own = nullptr;
    cudaError_t set(const void *src, size_t bytes, cudaStream_t s) {
        if (!src || on_device(src)) { d = src; return cudaSuccess; }
        cudaError_t e = cudaMalloc(&own, bytes);
        if (e != cudaSuccess) return e;
        d = own;
        return cudaMemcpyAsync(own, src, bytes, cudaMemcpyHostToDevice, s);
    }
    ~TmpIn() { if (own) cudaFree(own); }
};
struct TmpOut {
    void *d = nullptr, *own = nullptr, *host = nullptr;
    size_t bytes = 0;
    cudaError_t set(void *dst, size_t n) {
        if (!dst || on_device(dst)) { d = dst; return cudaSuccess; }
        cudaError_t e = cudaMalloc(&own, n);
        if (e != cudaSuccess) return e;
        d = own; host = dst; bytes = n;
        return cudaSuccess;
    }
    cudaError_t back(cudaStream_t s) { return host ? cudaMemcpyAsync(host, own, bytes, cudaMemcpyDeviceToHost, s) : cudaSuccess; }
    ~TmpOut() { if (own) cudaFree(own); }
};
} // namespace

extern "C" int kfpos_assemble_epochs(int device, int64_t n_logs, int64_t n_msgs, int n_anchors, const uint8_t *anchor,
                                     const uint8_t *seq, const int32_t *range_mm, const double *err, const double *t,
                                     int64_t max_epochs, int flags, double first_dt, int32_t *ranges_out,
                                     double *err_out, double *dt_out, int32_t *n_epochs, void *stream) {
    return kfpos_assemble_epochs_t(device, n_logs, n_msgs, n_anchors, anchor, seq, range_mm, err, t, max_epochs, flags,
                                   first_dt, ranges_out, err_out, dt_out, n_epochs, nullptr, stream);
}

extern "C" int kfpos_assemble_epochs_t(int device, int64_t n_logs, int64_t n_msgs, int n_anchors, const uint8_t *anchor,
                                       const uint8_t *seq, const int32_t *range_mm, const double *err, const double *t,
                                       int64_t max_epochs, int flags, double first_dt, int32_t *ranges_out,
                                       double *err_out, double *dt_out, int32_t *n_epochs, double *t_out, void *stream) {
    if (n_logs <= 0 || n_msgs < 0 || n_anchors <= 0 || n_anchors > KFPOS_MAX_ANCHORS || max_epochs <= 0)
        return KFPOS_ERR_INVALID;
    if (!anchor || !seq || !range_mm || !t || !ranges_out || !dt_out) return KFPOS_ERR_INVALID;
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count <= 0 || device < 0 || device >= count) {
        cudaGetLastError();
        return KFPOS_ERR_CUDA;
    }
    DeviceGuard g(device);
    if (!g.ok) return KFPOS_ERR_CUDA;
    cudaStream_t s = (cudaStream_t)stream;
    const size_t N = (size_t)n_logs, L = (size_t)n_msgs, M = (size_t)n_anchors, T = (size_t)max_epochs;
    TmpIn i_a, i_s, i_r, i_e, i_t;
    TmpOut o_r, o_e, o_dt, o_n, o_t;
    CK(i_a.set(anchor, L * N, s));
    CK(i_s.set(seq, L * N, s));
    CK(i_r.set(range_mm, 4 * L * N, s));
    CK(i_e.set(err, 8 * L * N, s));
    CK(i_t.set(t, 8 * L * N, s));
    CK(o_r.set(ranges_out, 4 * T * M * N));
    CK(o_e.set(err_out, 8 * T * M * N));
    CK(o_dt.set(dt_out, 8 * T * N));
    CK(o_n.set(n_epochs, 4 * N));
    CK(o_t.set(t_out, 8 * T * N));
    const int fix = (flags & KFPOS_ASM_FIX_ROW_CLEAR) ? 1 : 0;
    const size_t rows = fix ? 1 : 256;
    // the sequence-number table: per-device scratch that is kept between calls (grown on demand)
    static std::mutex mtx;
    static DevBuf tables[64][2];
    std::lock_guard<std::mutex> lock(mtx);
    DevBuf &tr = tables[device & 63][0], &te = tables[device & 63][1];
    CK(tr.reserve(4 * rows * M * N));
    CK(te.reserve(8 * rows * M * N));
    CK(cudaMemsetAsync(tr.p, 0xff, 4 * rows * M * N, s)); // initialiseTagList: -1
    CK(cudaMemsetAsync(te.p, 0, 8 * rows * M * N, s));
    AssembleParams p;
    p.N = n_logs; p.L = n_msgs; p.max_epochs = max_epochs;
    p.M = n_anchors; p.fix_b12 = fix; p.first_dt = first_dt;
    p.anchor = (const uint8_t *)i_a.d; p.seq = (const uint8_t *)i_s.d;
    p.range_mm = (const int32_t *)i_r.d; p.err = (const double *)i_e.d; p.t = (const double *)i_t.d;
    p.tbl_r = (int32_t *)tr.p; p.tbl_e = (double *)te.p;
    p.ranges_out = (int32_t *)o_r.d; p.err_out = (double *)o_e.d; p.dt_out = (double *)o_dt.d;
    p.n_epochs = (int32_t *)o_n.d;
    p.t_out = (double *)o_t.d;
    CK(launch_assemble(p, s));
    CK(o_t.back(s));
    CK(o_r.back(s));
    CK(o_e.back(s));
    CK(o_dt.back(s));
    CK(o_n.back(s));
    // temporary copies of host arrays are freed on return: finish the work first.  With device
    // pointers only, the call is asynchronous on `stream` like the rest of the API (the table
    // is reused by the next call on the same device, which is ordered behind this one only if it
    // uses the same stream: callers on different streams must synchronise themselves).
    if (i_a.own || i_s.own || i_r.own || i_e.own || i_t.own || o_r.own || o_e.own || o_dt.own || o_n.own || o_t.own)
        CK(cudaStreamSynchronize(s));
    return KFPOS_OK;
}

extern "C" int kfpos_merge_streams(int device, int64_t n_logs, int n_anchors, int64_t n_epochs, const double *t_epoch,
                                   const int32_t *ranges, const double *err, const int64_t n_samples[4],
                                   const double *const t_sensor[4], const double *const payload[4], int n_slots,
                                   const int32_t *slot_kind, double first_dt, const double *imu_aux,
                                   kfpos_event *events_out, double *dt_out, int32_t *ranges_out, double *err_out,
                                   double *sensors_out, int32_t *n_dropped, void *stream) {
    if (n_logs <= 0 || n_anchors <= 0 || n_anchors > KFPOS_MAX_ANCHORS || n_epochs < 0 || n_slots <= 0 || !slot_kind ||
        !dt_out)
        return KFPOS_ERR_INVALID;
    static const int rows_of[5] = {0, 5, 3, 2, 1};
    int64_t range_rows = 0, sensor_rows = 0;
    std::vector<int64_t> slot_row((size_t)n_slots);
    for (int sidx = 0; sidx < n_slots; ++sidx) {
        const int k = slot_kind[sidx];
        if (k < KFPOS_EV_TOA || k > KFPOS_EV_COMPASS) return KFPOS_ERR_INVALID;
        if (k == KFPOS_EV_TOA) {
            slot_row[sidx] = range_rows;
            range_rows += n_anchors;
        } else {
            slot_row[sidx] = sensor_rows;
            sensor_rows += rows_of[k];
        }
        if (events_out) {
            memset(&events_out[sidx], 0, sizeof(kfpos_event));
            events_out[sidx].kind = k;
            events_out[sidx].dt = 0.0; // the per-filter time steps replace it
            events_out[sidx].offset = slot_row[sidx];
            if (k == KFPOS_EV_IMU && imu_aux) memcpy(events_out[sidx].aux, imu_aux, sizeof(double) * 9);
        }
    }
    if ((range_rows > 0 && (!ranges_out || (n_epochs > 0 && (!t_epoch || !ranges)))) || (sensor_rows > 0 && !sensors_out))
        return KFPOS_ERR_INVALID;
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count <= 0 || device < 0 || device >= count) {
        cudaGetLastError();
        return KFPOS_ERR_CUDA;
    }
    DeviceGuard g(device);
    if (!g.ok) return KFPOS_ERR_CUDA;
    cudaStream_t s = (cudaStream_t)stream;
    const size_t N = (size_t)n_logs, M = (size_t)n_anchors;
    MergeParams p;
    memset(&p, 0, sizeof p);
    p.N = n_logs; p.M = n_anchors; p.n_slots = n_slots; p.first_dt = first_dt;
    TmpIn i_t[5], i_p[5], i_e, i_k, i_row;
    TmpOut o_dt, o_r, o_e, o_s, o_n;
    p.L[0] = n_epochs;
    CK(i_t[0].set(t_epoch, 8 * (size_t)n_epochs * N, s));
    CK(i_p[0].set(ranges, 4 * (size_t)n_epochs * M * N, s));
    CK(i_e.set(err, 8 * (size_t)n_epochs * M * N, s));
    p.t_src[0] = (const double *)i_t[0].d; p.ranges = (const int32_t *)i_p[0].d; p.err_src = (const double *)i_e.d;
    for (int k = 1; k < 5; ++k) {
        const int64_t Lk = n_samples ? n_samples[k - 1] : 0;
        if (Lk <= 0 || !t_sensor || !payload || !t_sensor[k - 1] || !payload[k - 1]) continue;
        p.L[k] = Lk;
        CK(i_t[k].set(t_sensor[k - 1], 8 * (size_t)Lk * N, s));
        CK(i_p[k].set(payload[k - 1], 8 * (size_t)Lk * rows_of[k] * N, s));
        p.t_src[k] = (const double *)i_t[k].d; p.src[k] = (const double *)i_p[k].d;
    }
    CK(i_k.set(nullptr, 0, s)); // (slot tables are small host arrays: always copied)
    int32_t *d_kind = nullptr;
    int64_t *d_row = nullptr;
    CK(cudaMalloc((void **)&d_kind, sizeof(int32_t) * (size_t)n_slots));
    cudaError_t e2 = cudaMalloc((void **)&d_row, sizeof(int64_t) * (size_t)n_slots);
    if (e2 != cudaSuccess) { cudaFree(d_kind); return map_cuda_err(e2); }
    auto cleanup = [&]() { cudaFree(d_kind); cudaFree(d_row); };
    auto fail = [&](cudaError_t e) { cudaStreamSynchronize(s); cleanup(); return map_cuda_err(e); };
    cudaError_t e = cudaMemcpyAsync(d_kind, slot_kind, sizeof(int32_t) * (size_t)n_slots, cudaMemcpyHostToDevice, s);
    if (e == cudaSuccess) e = cudaMemcpyAsync(d_row, slot_row.data(), sizeof(int64_t) * (size_t)n_slots, cudaMemcpyHostToDevice, s);
    if (e == cudaSuccess) e = o_dt.set(dt_out, 8 * (size_t)n_slots * N);
    if (e == cudaSuccess) e = o_r.set(ranges_out, 4 * (size_t)(range_rows > 0 ? range_rows : 1) * N);
    if (e == cudaSuccess) e = o_e.set(err_out, 8 * (size_t)(range_rows > 0 ? range_rows : 1) * N);
    if (e == cudaSuccess) e = o_s.set(sensors_out, 8 * (size_t)(sensor_rows > 0 ? sensor_rows : 1) * N);
    if (e == cudaSuccess) e = o_n.set(n_dropped, 4 * N);
    if (e != cudaSuccess) return fail(e);
    // slots nobody takes keep "no ranging" / zero payloads
    if (o_r.d) e = cudaMemsetAsync(o_r.d, 0xff, 4 * (size_t)(range_rows > 0 ? range_rows : 1) * N, s);
    if (e == cudaSuccess && o_e.d) e = cudaMemsetAsync(o_e.d, 0, 8 * (size_t)(range_rows > 0 ? range_rows : 1) * N, s);
    if (e == cudaSuccess && o_s.d) e = cudaMemsetAsync(o_s.d, 0, 8 * (size_t)(sensor_rows > 0 ? sensor_rows : 1) * N, s);
    if (e != cudaSuccess) return fail(e);
    p.slot_kind = d_kind; p.slot_row = d_row;
    p.dt_f = (double *)o_dt.d; p.ranges_out = (int32_t *)o_r.d; p.err_out = (double *)o_e.d;
    p.sensors_out = (double *)o_s.d; p.n_dropped = (int32_t *)o_n.d;
    e = launch_merge(p, s);
    if (e == cudaSuccess) e = o_dt.back(s);
    if (e == cudaSuccess) e = o_r.back(s);
    if (e == cudaSuccess) e = o_e.back(s);
    if (e == cudaSuccess) e = o_s.back(s);
    if (e == cudaSuccess) e = o_n.back(s);
    if (e != cudaSuccess) return fail(e);
    // the slot tables (and any staged host arrays) are freed on return: finish the work first
    e = cudaStreamSynchronize(s);
    cleanup();
    return e == cudaSuccess ? KFPOS_OK : map_cuda_err(e);
}

// ----------------------------------------------------------------- diagnostics
extern "C" int kfpos_batch_get_counters(kfpos_batch *b, double out[8], int reset, void *stream) {
    if (!b || !out) return KFPOS_ERR_INVALID;
    DeviceGuard g(b->device);
    cudaStream_t s = (cudaStream_t)stream;
    unsigned long long h[CNT_N];
    CK(cudaMemcpyAsync(h, b->d_counters, sizeof h, cudaMemcpyDeviceToHost, s));
    if (reset) CK(cudaMemsetAsync(b->d_counters, 0, sizeof h, s));
    CK(cudaStreamSynchronize(s));
    for (int i = 0; i < CNT_N; ++i) out[i] = (double)h[i];
    return KFPOS_OK;
}

extern "C" int kfpos_batch_set_truth(kfpos_batch *b, const double *truth, void *stream) {
    if (!b || b->model == KFPOS_MODEL_ML) return KFPOS_ERR_INVALID;
    DeviceGuard g(b->device);
    cudaStream_t s = (cudaStream_t)stream;
    b->partials_fresh = false;
    b->out4_valid = false;
    if (!truth) {
        b->d_truth = nullptr;
        return KFPOS_OK;
    }
    if (on_device(truth)) { // borrowed: the caller keeps it alive while it is registered
        b->d_truth = truth;
        return KFPOS_OK;
    }
    const size_t bytes = sizeof(double) * 3 * (size_t)b->N;
    if (!b->d_truth_own) CK(cudaMalloc((void **)&b->d_truth_own, bytes));
    CK(cudaMemcpyAsync(b->d_truth_own, truth, bytes, cudaMemcpyHostToDevice, s));
    CK(cudaStreamSynchronize(s));
    b->d_truth = b->d_truth_own;
    return KFPOS_OK;
}

namespace {
// leaves [sum |e|^2, sum |e_xy|^2, n, n_bad] of this batch in d_out4.  truth == null: the partials the last
// replay launch left behind (kfpos_batch_set_truth) are folded; otherwise they are computed first.
int enqueue_error_stats(kfpos_batch *b, const double *truth, cudaStream_t s) {
    const void *d_truth = nullptr;
    if (truth) {
        int rc = stage_in(b, 0, truth, sizeof(double) * 3 * (size_t)b->N, s, &d_truth);
        if (rc) return rc;
    } else if (!b->partials_fresh) {
        if (!b->d_truth) return KFPOS_ERR_NOT_READY;
        d_truth = b->d_truth; // registered, but the state changed since the last replay (single steps, set_state)
    }
    // K8 is planar: z is the configured tag height (KF.cpp:328-332)
    CK(launch_error_stats(b->N, b->d_x, b->model == KFPOS_MODEL_K8 ? -1 : 2, b->cfg.fixed_height, b->d_status,
                          (const double *)d_truth, b->d_partials, b->d_out4, s));
    b->partials_fresh = false; // the tree folds the partials in place
    b->out4_valid = true;
    return KFPOS_OK;
}

// NCCL is bound at run time (dlopen): the library loads and every other entry point works on a machine
// without it, and inside a process that already holds a copy (PyTorch's) that copy is the one used.
typedef int (*nccl_allgather_fn)(const void *, void *, size_t, int, void *, cudaStream_t);
typedef int (*nccl_count_fn)(void *, int *);
struct NcclApi {
    nccl_allgather_fn all_gather = nullptr;
    nccl_count_fn count = nullptr, user_rank = nullptr;
    bool tried = false;
};
NcclApi &nccl_api() {
    static NcclApi api;
    if (!api.tried) {
        api.tried = true;
        void *h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
        if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
        if (h) {
            api.all_gather = (nccl_allgather_fn)dlsym(h, "ncclAllGather");
            api.count = (nccl_count_fn)dlsym(h, "ncclCommCount");
            api.user_rank = (nccl_count_fn)dlsym(h, "ncclCommUserRank");
        }
    }
    return api;
}
} // namespace

extern "C" int kfpos_batch_error_stats(kfpos_batch *b, const double *truth, double out[4], void *stream) {
    if (!b || b->model == KFPOS_MODEL_ML) return KFPOS_ERR_INVALID;
    DeviceGuard g(b->device);
    cudaStream_t s = (cudaStream_t)stream;
    int rc = enqueue_error_stats(b, truth, s);
    if (rc) return rc;
    if (out) { // out == null: enqueue only, the result stays on the device (kfpos_stats_allreduce reads it)
        CK(cudaMemcpyAsync(out, b->d_out4, sizeof(double) * 4, cudaMemcpyDeviceToHost, s));
        CK(cudaStreamSynchronize(s));
    }
    return KFPOS_OK;
}

extern "C" int kfpos_stats_allreduce(kfpos_batch *b, struct ncclComm *comm, const double *truth, double out[6],
                                     void *stream) {
    if (!b || b->model == KFPOS_MODEL_ML || !out) return KFPOS_ERR_INVALID;
    DeviceGuard g(b->device);
    cudaStream_t s = (cudaStream_t)stream;
    // truth == null: what the last kfpos_batch_error_stats left on the device, if the state has not changed since
    if (truth || !b->out4_valid) {
        int rc = enqueue_error_stats(b, truth, s);
        if (rc) return rc;
    }
    const double *d_res = b->d_out4;
    if (comm) {
        NcclApi &api = nccl_api();
        if (!api.all_gather || !api.count) return KFPOS_ERR_UNSUPPORTED;
        int n_ranks = 0;
        if (api.count(comm, &n_ranks) != 0 || n_ranks < 1 || n_ranks > 1024) return KFPOS_ERR_INVALID;
        // ONE collective: every rank's 4 doubles to every rank (ncclDouble = 8), then the same pairwise
        // tree over the rank index on every rank -- the top levels of the global tree, in a fixed order
        if (api.all_gather(b->d_out4, b->d_gather, 4, 8, comm, s) != 0) return KFPOS_ERR_CUDA;
        CK(launch_error_stats_tree(n_ranks, b->d_gather, b->d_gather, s));
        d_res = b->d_gather;
    }
    CK(cudaMemcpyAsync(out, d_res, sizeof(double) * 4, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    const double n = out[2] > 1.0 ? out[2] : 1.0;
    out[4] = sqrt(out[0] / n);
    out[5] = sqrt(out[1] / n);
    return KFPOS_OK;
}

// ------------------------------------------------------- per-epoch statistics
extern "C" int kfpos_batch_set_truth_traj(kfpos_batch *b, int64_t n_rows, const double *truth, void *stream) {
    if (!b || b->model == KFPOS_MODEL_ML || (truth && n_rows <= 0)) return KFPOS_ERR_INVALID;
    DeviceGuard g(b->device);
    cudaStream_t s = (cudaStream_t)stream;
    // (cudaFree waits for the device: no launch still reads the buffers of the previous registration)
    cudaFree(b->d_etruth_own);
    cudaFree(b->d_escratch);
    cudaFree(b->d_efold);
    cudaFree(b->d_eout);
    b->d_etruth_own = b->d_escratch = b->d_efold = b->d_eout = nullptr;
    b->d_etruth = nullptr;
    b->es_rows = b->es_cursor = b->es_fold_rows = 0;
    if (!truth) return KFPOS_OK;
    const int64_t W = es_warps(b);
    const size_t row_bytes = sizeof(double) * ES_W * (size_t)W;
    // the fold of kfpos_batch_epoch_stats works on batches of rows in a buffer of at most 256 MB
    int64_t fold_rows = (int64_t)(((size_t)256 << 20) / row_bytes);
    if (fold_rows < 1) fold_rows = 1;
    if (fold_rows > n_rows) fold_rows = n_rows;
    const bool dev = on_device(truth);
    cudaError_t e = cudaMalloc((void **)&b->d_escratch, row_bytes * (size_t)n_rows);
    if (e == cudaSuccess) e = cudaMalloc((void **)&b->d_efold, row_bytes * (size_t)fold_rows);
    if (e == cudaSuccess) e = cudaMalloc((void **)&b->d_eout, sizeof(double) * ES_W * (size_t)n_rows);
    const size_t tbytes = sizeof(double) * 3 * (size_t)b->N * (size_t)n_rows;
    if (e == cudaSuccess && !dev) e = cudaMalloc((void **)&b->d_etruth_own, tbytes);
    if (e == cudaSuccess && !dev) e = cudaMemcpyAsync(b->d_etruth_own, truth, tbytes, cudaMemcpyHostToDevice, s);
    if (e == cudaSuccess && !dev) e = cudaStreamSynchronize(s);
    if (e != cudaSuccess) {
        cudaFree(b->d_etruth_own);
        cudaFree(b->d_escratch);
        cudaFree(b->d_efold);
        cudaFree(b->d_eout);
        b->d_etruth_own = b->d_escratch = b->d_efold = b->d_eout = nullptr;
        cudaGetLastError();
        return map_cuda_err(e);
    }
    b->d_etruth = dev ? truth : b->d_etruth_own; // a device array is borrowed: the caller keeps it alive
    b->es_rows = n_rows;
    b->es_fold_rows = fold_rows;
    return KFPOS_OK;
}

namespace {
// [n_rows][6] of this batch into the device array `d_out`: rows [0, cursor) folded over the warp index (batches
// of es_fold_rows rows through d_efold, the per-warp sums stay as they are), the rest zero
int enqueue_epoch_stats(kfpos_batch *b, double *d_out, cudaStream_t s) {
    const int64_t W = es_warps(b), done = b->es_cursor < b->es_rows ? b->es_cursor : b->es_rows;
    for (int64_t r0 = 0; r0 < done; r0 += b->es_fold_rows) {
        const int64_t rb = done - r0 < b->es_fold_rows ? done - r0 : b->es_fold_rows;
        CK(launch_stats_tree(ES_W, rb, W, b->d_escratch + r0 * W * ES_W, b->d_efold, W * ES_W, ES_W, d_out + r0 * ES_W, s));
    }
    if (done < b->es_rows)
        CK(cudaMemsetAsync(d_out + done * ES_W, 0, sizeof(double) * ES_W * (size_t)(b->es_rows - done), s));
    return KFPOS_OK;
}
int es_ready(const kfpos_batch *b, int64_t n_rows, const double *out) {
    if (!b || b->model == KFPOS_MODEL_ML || !out) return KFPOS_ERR_INVALID;
    if (!b->d_escratch) return KFPOS_ERR_NOT_READY;
    return n_rows == b->es_rows ? KFPOS_OK : KFPOS_ERR_INVALID;
}
} // namespace

extern "C" int kfpos_batch_epoch_stats(kfpos_batch *b, int64_t n_rows, double *out, void *stream) {
    int rc = es_ready(b, n_rows, out);
    if (rc) return rc;
    DeviceGuard g(b->device);
    cudaStream_t s = (cudaStream_t)stream;
    const bool dev = on_device(out);
    if ((rc = enqueue_epoch_stats(b, dev ? out : b->d_eout, s))) return rc;
    if (!dev) {
        CK(cudaMemcpyAsync(out, b->d_eout, sizeof(double) * ES_W * (size_t)n_rows, cudaMemcpyDeviceToHost, s));
        CK(cudaStreamSynchronize(s));
    }
    return KFPOS_OK;
}

extern "C" int kfpos_epoch_stats_allreduce(kfpos_batch *b, struct ncclComm *comm, int64_t n_rows, double *out,
                                           void *stream) {
    int rc = es_ready(b, n_rows, out);
    if (rc) return rc;
    DeviceGuard g(b->device);
    cudaStream_t s = (cudaStream_t)stream;
    if ((rc = enqueue_epoch_stats(b, b->d_eout, s))) return rc;
    const double *d_res = b->d_eout;
    const size_t bytes = sizeof(double) * ES_W * (size_t)n_rows;
    if (comm) {
        NcclApi &api = nccl_api();
        if (!api.all_gather || !api.count) return KFPOS_ERR_UNSUPPORTED;
        int n_ranks = 0;
        if (api.count(comm, &n_ranks) != 0 || n_ranks < 1 || n_ranks > 1024) return KFPOS_ERR_INVALID;
        CK(b->es_gather.reserve(bytes * (size_t)n_ranks));
        double *gat = (double *)b->es_gather.p;
        // ONE collective: every rank's [n_rows][6] to every rank ([rank][row][6]), then per row the pairwise tree
        // over the rank index -- the top levels of the global tree; row r's result lands on its rank-0 entry
        if (api.all_gather(b->d_eout, gat, (size_t)n_rows * ES_W, 8, comm, s) != 0) return KFPOS_ERR_CUDA;
        CK(launch_stats_tree(ES_W, n_rows, n_ranks, gat, gat, ES_W, n_rows * ES_W, gat, s));
        d_res = gat;
    }
    const bool dev = on_device(out);
    CK(cudaMemcpyAsync(out, d_res, bytes, dev ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost, s));
    if (!dev) CK(cudaStreamSynchronize(s));
    return KFPOS_OK;
}

extern "C" int kfpos_measure_fp64_peak(int device, double *flops_per_s) {
    if (!flops_per_s) return KFPOS_ERR_INVALID;
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || device < 0 || device >= count) {
        cudaGetLastError();
        return KFPOS_ERR_CUDA;
    }
    DeviceGuard g(device);
    if (!g.ok) return KFPOS_ERR_CUDA;
    CK(measure_fp64_peak(flops_per_s));
    return KFPOS_OK;
}

extern "C" int kfpos_synth_k8(int device, int64_t n_filters, int64_t first_filter, uint64_t seed, int n_anchors,
                              const double *anchors_xyz, double tag_z, double sigma_r, int n_events,
                              const kfpos_synth_event *events, double t_end, int64_t range_rows, int64_t sensor_rows,
                              int32_t *ranges, double *sensors, double *x0, double *truth_end, void *stream) {
    static_assert(sizeof(kfpos_synth_event) == sizeof(SynthEvent), "kfpos_synth_event and SynthEvent must have one layout");
    if (n_filters <= 0 || n_anchors <= 0 || n_anchors > KFPOS_MAX_ANCHORS || !anchors_xyz || n_events < 0 ||
        (n_events > 0 && !events) || range_rows < 0 || sensor_rows < 0)
        return KFPOS_ERR_INVALID;
    for (int i = 0; i < n_events; ++i) { // every event must write inside the tensors it was given
        const int rows = events[i].kind == KFPOS_EV_TOA ? n_anchors
                         : events[i].kind == KFPOS_EV_PX4 ? 5 : events[i].kind == KFPOS_EV_IMU ? 3
                         : events[i].kind == KFPOS_EV_COMPASS ? 1 : -1;
        const int64_t lim = events[i].kind == KFPOS_EV_TOA ? range_rows : sensor_rows;
        if (rows < 0 || events[i].offset < 0 || events[i].offset + rows > lim) return KFPOS_ERR_INVALID;
        if ((events[i].kind == KFPOS_EV_TOA && !ranges) || (events[i].kind != KFPOS_EV_TOA && !sensors))
            return KFPOS_ERR_INVALID;
    }
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count <= 0 || device < 0 || device >= count) {
        cudaGetLastError();
        return KFPOS_ERR_CUDA;
    }
    DeviceGuard g(device);
    if (!g.ok) return KFPOS_ERR_CUDA;
    cudaStream_t s = (cudaStream_t)stream;
    const size_t N = (size_t)n_filters;
    TmpOut o_r, o_s, o_x, o_t;
    CK(o_r.set(ranges, 4 * (size_t)range_rows * N));
    CK(o_s.set(sensors, 8 * (size_t)sensor_rows * N));
    CK(o_x.set(x0, 8 * 8 * N));
    CK(o_t.set(truth_end, 8 * 3 * N));
    // the schedule goes through a small per-device ring of scratch buffers (a pageable source has left the caller's
    // array when cudaMemcpyAsync returns): with device outputs the call is then asynchronous on `stream`, so that a
    // caller can generate chunk c + 1 on one stream while chunk c is replayed on another
    void *d_ev = nullptr;
    if (n_events > 0) {
        static std::mutex mtx;
        static DevBuf ring[64][8];
        static unsigned next[64];
        std::lock_guard<std::mutex> lock(mtx);
        DevBuf &slot = ring[device & 63][next[device & 63]++ & 7];
        if (slot.cap < sizeof(SynthEvent) * (size_t)n_events) {
            CK(cudaStreamSynchronize(s)); // growing a slot frees the old one: nothing may still read it
            CK(cudaDeviceSynchronize());
            CK(slot.reserve(sizeof(SynthEvent) * (size_t)(n_events < 256 ? 256 : n_events)));
        }
        d_ev = slot.p;
        CK(cudaMemcpyAsync(d_ev, events, sizeof(SynthEvent) * (size_t)n_events, cudaMemcpyHostToDevice, s));
    }
    SynthK8Params p;
    memset(&p.anchors, 0, sizeof p.anchors);
    p.anchors.n = n_anchors;
    for (int i = 0; i < n_anchors; ++i) {
        p.anchors.x[i] = anchors_xyz[3 * i]; p.anchors.y[i] = anchors_xyz[3 * i + 1]; p.anchors.z[i] = anchors_xyz[3 * i + 2];
    }
    p.N = n_filters; p.filter0 = first_filter; p.seed = seed; p.M = n_anchors; p.n_events = n_events;
    p.tag_z = tag_z; p.sigma_r = sigma_r; p.t_end = t_end;
    p.events = (const SynthEvent *)d_ev;
    p.ranges = (int32_t *)o_r.d; p.sensors = (double *)o_s.d; p.x0 = (double *)o_x.d; p.truth_end = (double *)o_t.d;
    cudaError_t e = launch_synth_k8(p, s);
    if (e == cudaSuccess) e = o_r.back(s);
    if (e == cudaSuccess) e = o_s.back(s);
    if (e == cudaSuccess) e = o_x.back(s);
    if (e == cudaSuccess) e = o_t.back(s);
    if (e != cudaSuccess) return map_cuda_err(e);
    // host staging is freed on return: finish the work first; device outputs: asynchronous on `stream`
    if (o_r.own || o_s.own || o_x.own || o_t.own) CK(cudaStreamSynchronize(s));
    return KFPOS_OK;
}

extern "C" int kfpos_synth_k8_truth(int device, int64_t n_filters, int64_t first_filter, uint64_t seed, int n_times,
                                    const double *t, double tag_z, double *truth, void *stream) {
    if (n_filters <= 0 || n_times < 0 || (n_times > 0 && (!t || !truth))) return KFPOS_ERR_INVALID;
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count <= 0 || device < 0 || device >= count) {
        cudaGetLastError();
        return KFPOS_ERR_CUDA;
    }
    if (n_times == 0) return KFPOS_OK;
    DeviceGuard g(device);
    if (!g.ok) return KFPOS_ERR_CUDA;
    cudaStream_t s = (cudaStream_t)stream;
    TmpIn i_t;
    TmpOut o_t;
    CK(i_t.set(t, sizeof(double) * (size_t)n_times, s));
    CK(o_t.set(truth, sizeof(double) * 3 * (size_t)n_filters * (size_t)n_times));
    SynthTruthParams p;
    p.N = n_filters; p.filter0 = first_filter; p.seed = seed; p.n_times = n_times; p.tag_z = tag_z;
    p.t = (const double *)i_t.d;
    p.truth = (double *)o_t.d;
    CK(launch_synth_k8_truth(p, s));
    CK(o_t.back(s));
    // staging is freed on return: finish the work first; device arrays only: asynchronous on `stream`
    if (i_t.own || o_t.own) CK(cudaStreamSynchronize(s));
    return KFPOS_OK;
}

extern "C" int kfpos_synth_toa_ranges(int device, int64_t n_filters, int n_anchors, const double *anchors_xyz,
                                      int n_epochs, const double *t, const kfpos_synth_toa *gen, int fmt,
                                      void *ranges, void *stream) {
    const auto prob = [](double q) { return q >= 0.0 && q <= 1.0; }; // false for NaN
    if (n_filters <= 0 || n_anchors <= 0 || n_anchors > KFPOS_MAX_ANCHORS || !anchors_xyz || n_epochs < 0 ||
        (n_epochs > 0 && (!t || !ranges)) || !gen || (fmt != KFPOS_FMT_I32_MM && fmt != KFPOS_FMT_U16_MM))
        return KFPOS_ERR_INVALID;
    if (!prob(gen->p_missing) || !prob(gen->p_nlos) || !(gen->sigma_r >= 0.0) ||
        (gen->p_nlos > 0.0 && !(gen->nlos_mean > 0.0)) || gen->first_filter < 0 || gen->first_epoch < 0 ||
        gen->first_epoch + n_epochs > (int64_t)0xFFFFFFFF) // epoch index 0xFFFFFFFF: the per-filter constants
        return KFPOS_ERR_INVALID;
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count <= 0 || device < 0 || device >= count) {
        cudaGetLastError();
        return KFPOS_ERR_CUDA;
    }
    if (n_epochs == 0) return KFPOS_OK;
    DeviceGuard g(device);
    if (!g.ok) return KFPOS_ERR_CUDA;
    cudaStream_t s = (cudaStream_t)stream;
    const size_t row = fmt_size(fmt) * (size_t)n_anchors * (size_t)n_filters; // bytes of one epoch
    TmpOut o_r;
    CK(o_r.set(ranges, row * (size_t)n_epochs));
    // the epoch times travel in the parameter block, SYNTH_TOA_T per launch: nothing to stage, so a device
    // `ranges` leaves the call asynchronous (the next chunk can be generated while this one is replayed)
    SynthToaParams p{};
    p.anchors.n = n_anchors;
    for (int i = 0; i < n_anchors; ++i) {
        p.anchors.x[i] = anchors_xyz[3 * i]; p.anchors.y[i] = anchors_xyz[3 * i + 1]; p.anchors.z[i] = anchors_xyz[3 * i + 2];
    }
    p.N = n_filters; p.filter0 = gen->first_filter; p.seed = gen->seed; p.M = n_anchors;
    p.tag_z = gen->tag_z; p.sigma_r = gen->sigma_r; p.p_missing = gen->p_missing; p.p_nlos = gen->p_nlos;
    p.nlos_mean = gen->nlos_mean;
    for (int k0 = 0; k0 < n_epochs; k0 += SYNTH_TOA_T) {
        p.n_epochs = n_epochs - k0 < SYNTH_TOA_T ? n_epochs - k0 : SYNTH_TOA_T;
        p.epoch0 = (uint32_t)(gen->first_epoch + k0);
        memcpy(p.t, t + k0, sizeof(double) * (size_t)p.n_epochs);
        p.ranges = (char *)o_r.d + row * (size_t)k0;
        CK(launch_synth_toa(p, fmt == KFPOS_FMT_U16_MM, s));
    }
    CK(o_r.back(s));
    // host staging is freed on return: finish the work first; device output: asynchronous on `stream`
    if (o_r.own) CK(cudaStreamSynchronize(s));
    return KFPOS_OK;
}

extern "C" int kfpos_selftest_math(int device, int64_t n, const double *x, double *rcp, double *rsqrt, double *sn,
                                   double *cs) {
    if (n <= 0 || !x) return KFPOS_ERR_INVALID;
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count <= 0 || device < 0 || device >= count) {
        cudaGetLastError();
        return KFPOS_ERR_CUDA;
    }
    DeviceGuard g(device);
    if (!g.ok) return KFPOS_ERR_CUDA;
    TmpIn i_x;
    TmpOut o[4];
    double *outs[4] = {rcp, rsqrt, sn, cs};
    CK(i_x.set(x, 8 * (size_t)n, nullptr));
    for (int k = 0; k < 4; ++k) CK(o[k].set(outs[k], 8 * (size_t)n));
    CK(launch_selftest_math(n, (const double *)i_x.d, (double *)o[0].d, (double *)o[1].d, (double *)o[2].d,
                            (double *)o[3].d, nullptr));
    for (int k = 0; k < 4; ++k) CK(o[k].back(nullptr));
    CK(cudaStreamSynchronize(nullptr));
    return KFPOS_OK;
}

extern "C" int kfpos_selftest_ieee(int device, int64_t n, const double *a, const double *b, double *div_fast,
                                   double *div_ieee, double *sqrt_fast, double *sqrt_ieee, int32_t *flags) {
    if (n <= 0 || !a || !b) return KFPOS_ERR_INVALID;
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count <= 0 || device < 0 || device >= count) {
        cudaGetLastError();
        return KFPOS_ERR_CUDA;
    }
    DeviceGuard g(device);
    if (!g.ok) return KFPOS_ERR_CUDA;
    TmpIn i_a, i_b;
    TmpOut o[4], o_f;
    double *outs[4] = {div_fast, div_ieee, sqrt_fast, sqrt_ieee};
    CK(i_a.set(a, 8 * (size_t)n, nullptr));
    CK(i_b.set(b, 8 * (size_t)n, nullptr));
    for (int k = 0; k < 4; ++k) CK(o[k].set(outs[k], 8 * (size_t)n));
    CK(o_f.set(flags, 4 * (size_t)n));
    CK(launch_selftest_ieee(n, (const double *)i_a.d, (const double *)i_b.d, (double *)o[0].d, (double *)o[1].d,
                            (double *)o[2].d, (double *)o[3].d, (int32_t *)o_f.d, nullptr));
    for (int k = 0; k < 4; ++k) CK(o[k].back(nullptr));
    CK(o_f.back(nullptr));
    CK(cudaStreamSynchronize(nullptr));
    return KFPOS_OK;
}
