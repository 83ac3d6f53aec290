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
    DevBuf gather; // [n_ranks][4] of kfpos_stats_allreduce
    // per-epoch statistics (kfpos_batch_set_truth_traj): truth rows SoA [es_rows][3][N], per-warp sums
    // [es_rows][n_warps][6] left by the replay kernels, the next output row, and the fold buffers
    const double *d_etruth = nullptr;
    double *d_etruth_own = nullptr, *d_escratch = nullptr, *d_efold = nullptr, *d_eout = nullptr;
    int64_t es_rows = 0, es_cursor = 0, es_fold_rows = 0;
    DevBuf es_gather;
    // per-epoch error histogram (kfpos_batch_set_error_hist): the quantity, the device edge table [EH_MAX_BINS - 1]
    // (squared for the error quantities, +inf behind the last edge), and the counts [es_rows][eh_bins], which
    // exist while a truth trajectory is registered too
    int eh_quantity = 0, eh_bins = 0; // eh_bins == 0: no histogram
    double *d_eh_edges = nullptr;
    unsigned long long *d_eh_counts = nullptr;
    DevBuf eh_gather;
    DevBuf crlb; // per-warp partials of kfpos_batch_crlb, [rows][n_warps][4], at most 256 MB
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

// Argument staging of one call.  Device pointers pass through; a host data array goes through a device buffer,
// and then the call synchronises its stream before returning (include/kfpos_b200.h, Conventions).  The buffers of
// a call on a batch are the slots of its scratch pool, taken one after the other in the order the call asks for
// them, so two buffers of one call never alias; a call without a handle allocates its own and frees them on return.
// Errors are sticky: after a failed step every later one is skipped and `rc` holds the first error, which the
// caller checks before it launches anything that reads the buffers.
class Staging {
  public:
    int rc = KFPOS_OK;
    bool sync = false; // finish() synchronises: a host data array was read or written, or a buffer is freed on return

    Staging(kfpos_batch *b, cudaStream_t s) : pool_(b->scratch), s_(s) {}
    explicit Staging(cudaStream_t s) : s_(s) {}
    Staging(const Staging &) = delete;
    Staging &operator=(const Staging &) = delete;
    ~Staging() {
        for (void *p : own_) cudaFree(p);
    }

    // a device array for the call's own intermediates
    template <class T = void> T *buf(size_t bytes) { return static_cast<T *>(alloc(bytes)); }
    // a data array the call reads
    template <class T> const T *in(const T *p, size_t bytes) {
        if (!p || on_device(p)) return p;
        T *d = buf<T>(bytes);
        copy(d, p, bytes, cudaMemcpyHostToDevice);
        sync = true;
        return d;
    }
    // a data array the call writes: a host array gets a device buffer that finish() copies back
    template <class T> T *out(T *p, size_t bytes) {
        if (!p || on_device(p)) return p;
        T *d = buf<T>(bytes);
        if (d) back_.push_back({p, d, bytes});
        sync = true;
        return d;
    }
    // a small control array (the ones the header declares as HOST arrays: time steps, event schedules, slot
    // tables), always copied.  It does not make the call synchronise: a copy from pageable memory has left the
    // caller's array when cudaMemcpyAsync returns.
    template <class T> const T *ctl(const T *p, size_t bytes) {
        T *d = buf<T>(bytes);
        copy(d, p, bytes, on_device(p) ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice);
        return d;
    }
    // direct copies between a caller's data array and batch memory; a null array is skipped
    void copy_in(void *dst_dev, const void *src, size_t bytes) {
        if (!src) return;
        const bool host = !on_device(src);
        copy(dst_dev, src, bytes, host ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice);
        sync = sync || host;
    }
    void copy_out(void *dst, const void *src_dev, size_t bytes) {
        if (!dst) return;
        const bool host = !on_device(dst);
        copy(dst, src_dev, bytes, host ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice);
        sync = sync || host;
    }
    // enqueues the copy-backs of out(), synchronises if `sync`, and returns the status of the call
    int finish() {
        for (const Back &c : back_) copy(c.host, c.dev, c.bytes, cudaMemcpyDeviceToHost);
        if (sync && rc == KFPOS_OK) fail(cudaStreamSynchronize(s_));
        return rc;
    }

  private:
    struct Back {
        void *host;
        const void *dev;
        size_t bytes;
    };
    DevBuf *pool_ = nullptr;
    int next_ = 0;
    cudaStream_t s_;
    std::vector<void *> own_;
    std::vector<Back> back_;

    void fail(cudaError_t e) {
        if (e != cudaSuccess && rc == KFPOS_OK) rc = map_cuda_err(e);
    }
    void copy(void *dst, const void *src, size_t bytes, cudaMemcpyKind kind) {
        if (rc == KFPOS_OK) fail(cudaMemcpyAsync(dst, src, bytes, kind, s_));
    }
    void *alloc(size_t bytes) {
        if (rc != KFPOS_OK) return nullptr;
        if (!pool_) {
            void *p = nullptr;
            fail(cudaMalloc(&p, bytes));
            if (p) own_.push_back(p);
            sync = true; // freed on return: the work that uses it has to be done by then
            return p;
        }
        if (next_ == N_SCRATCH) { // N_SCRATCH covers the call with the most buffers, kfpos_batch_ml_solve
            rc = KFPOS_ERR_NOMEM;
            return nullptr;
        }
        DevBuf &d = pool_[next_++];
        fail(d.reserve(bytes));
        return rc == KFPOS_OK ? d.p : nullptr;
    }
};

// KFPOS_ERR_CUDA unless `device` is a CUDA device of this process
int check_device(int device) {
    int count = 0;
    if (cudaGetDeviceCount(&count) == cudaSuccess && device >= 0 && device < count) return KFPOS_OK;
    cudaGetLastError();
    return KFPOS_ERR_CUDA;
}

// reads `bytes` of a host or device array on the host
int to_host(void *dst, const void *src, size_t bytes) {
    if (on_device(src)) CK(cudaMemcpy(dst, src, bytes, cudaMemcpyDeviceToHost));
    else memcpy(dst, src, bytes);
    return KFPOS_OK;
}

// the anchor table of `n` (x, y, z) triples in a host or device array
int anchor_table(int n, const double *xyz, AnchorTable *t) {
    double host[3 * KFPOS_MAX_ANCHORS];
    int rc = to_host(host, xyz, sizeof(double) * 3 * (size_t)n);
    if (rc) return rc;
    memset(t, 0, sizeof *t);
    for (int i = 0; i < n; ++i) {
        t->x[i] = host[3 * i];
        t->y[i] = host[3 * i + 1];
        t->z[i] = host[3 * i + 2];
    }
    t->n = n;
    return KFPOS_OK;
}

size_t fmt_size(int fmt) { return fmt == KFPOS_FMT_F64_M ? 8 : (fmt == KFPOS_FMT_I32_MM ? 4 : 2); }
bool fmt_ok(int fmt) { return fmt >= KFPOS_FMT_F64_M && fmt <= KFPOS_FMT_U16_MM; }

// rows of N values one event writes or reads in its log: the M rangings of a TOA event, the payload rows of a
// sensor event (header, kfpos_event); -1 for an unknown kind
int event_rows(int kind, int M) {
    static const int payload[5] = {0, 5, 3, 2, 1}; // -, PX4, IMU, MAG, COMPASS
    if (kind < KFPOS_EV_TOA || kind > KFPOS_EV_COMPASS) return -1;
    return kind == KFPOS_EV_TOA ? M : payload[kind];
}

// T epochs of a [T][M][N] range log as a K8 / T9 schedule of TOA events; dt null: the time steps are per filter
std::vector<kfpos_event> toa_schedule(size_t T, size_t M, const double *dt) {
    std::vector<kfpos_event> evs(T); // zero-initialised
    for (size_t t = 0; t < T; ++t) {
        evs[t].kind = KFPOS_EV_TOA;
        evs[t].dt = dt ? dt[t] : 0.0;
        evs[t].offset = (int64_t)(t * M);
    }
    return evs;
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
// the per-epoch statistics pointers of the next launch, then the cursor moves past its `rows` output rows.  The
// histogram rows of the launch are zeroed first: a re-run after set_state overwrites them, as it does the sums.
template <class Params>
int es_bind(kfpos_batch *b, Params &p, int64_t rows, cudaStream_t s) {
    p.n_warps = es_warps(b);
    p.etruth = nullptr;
    p.escratch = nullptr;
    p.ehist = nullptr;
    p.eedges = b->d_eh_edges;
    p.equantity = b->eh_quantity;
    p.ebins = b->eh_bins;
    if (!b->d_escratch) return KFPOS_OK;
    p.etruth = b->d_etruth + b->es_cursor * 3 * b->N;
    p.escratch = b->d_escratch + b->es_cursor * p.n_warps * ES_W;
    if (b->d_eh_counts) {
        p.ehist = b->d_eh_counts + b->es_cursor * b->eh_bins;
        CK(cudaMemsetAsync(p.ehist, 0, sizeof(unsigned long long) * (size_t)rows * (size_t)b->eh_bins, s));
    }
    b->es_cursor += rows;
    return KFPOS_OK;
}

// the fields the T6, K8 and T9 replay parameters share (kept apart in each struct: a shared sub-struct would move
// the kernel parameter offsets); the launch has `rows` output rows
template <class Params>
int bind_replay(kfpos_batch *b, Params &p, const RangeStream &rs, const double *dt_f, double *traj, int64_t rows,
                cudaStream_t s) {
    p.anchors = b->anchors;
    p.rs = rs;
    p.N = b->N;
    p.x = b->d_x;
    p.P = b->d_P;
    p.status = b->d_status;
    p.dt_f = dt_f;
    p.traj = traj;
    p.counters = b->d_counters;
    p.truth = b->d_truth;
    p.partials = b->d_partials;
    return es_bind(b, p, rows, s);
}

// after a replay launch: the partials of a registered truth are those of the new state, the folded statistics are
// stale, and (K8 / T9) the latched IMU covariances the launch wrote move to where the next launch reads them
int replayed(kfpos_batch *b, cudaStream_t s) {
    if (b->d_latch_u)
        CK(cudaMemcpyAsync(b->d_latch_u, b->d_latch_u + 16, sizeof(double) * 16, cudaMemcpyDeviceToDevice, s));
    b->partials_fresh = b->d_truth != nullptr;
    b->out4_valid = false;
    return KFPOS_OK;
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
    if (int rc = check_device(device)) return rc;
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
        if (e == cudaSuccess) e = b->gather.reserve(sizeof(double) * 4 * 1024);
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
    b->gather.release();
    cudaFree(b->d_etruth_own);
    cudaFree(b->d_escratch);
    cudaFree(b->d_efold);
    cudaFree(b->d_eout);
    b->es_gather.release();
    cudaFree(b->d_eh_edges);
    cudaFree(b->d_eh_counts);
    b->eh_gather.release();
    b->crlb.release();
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
    DeviceGuard g(b->device);
    AnchorTable t;
    int rc = anchor_table(n_anchors, xyz, &t);
    if (rc) return rc;
    b->anchors = t;
    b->have_anchors = true;
    return KFPOS_OK;
}

extern "C" int kfpos_batch_set_state(kfpos_batch *b, const double *x, const double *P, void *stream) {
    if (!b || b->model == KFPOS_MODEL_ML || !x) return KFPOS_ERR_INVALID;
    DeviceGuard g(b->device);
    cudaStream_t s = (cudaStream_t)stream;
    const size_t N = (size_t)b->N;
    Staging st(b, s);
    st.copy_in(b->d_x, x, sizeof(double) * b->n * N);
    const double *d_P = st.in(P, sizeof(double) * b->n * b->n * N);
    if (st.rc) return st.rc;
    if (d_P) {
        CK(launch_pack_cov(b->n, b->N, d_P, b->d_P, s));
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
    return st.finish();
}

extern "C" int kfpos_batch_get_latches(kfpos_batch *b, double *latch, int32_t *has, double *latch_u, void *stream) {
    if (!b || !b->d_latch) return KFPOS_ERR_INVALID;
    DeviceGuard g(b->device);
    const size_t N = (size_t)b->N;
    Staging st(b, (cudaStream_t)stream);
    st.copy_out(latch, b->d_latch, sizeof(double) * 16 * N);
    st.copy_out(has, b->d_has, sizeof(int32_t) * N);
    st.copy_out(latch_u, b->d_latch_u, sizeof(double) * 16);
    return st.finish();
}

extern "C" int kfpos_batch_set_latches(kfpos_batch *b, const double *latch, const int32_t *has, const double *latch_u,
                                       void *stream) {
    if (!b || !b->d_latch) return KFPOS_ERR_INVALID;
    DeviceGuard g(b->device);
    const size_t N = (size_t)b->N;
    Staging st(b, (cudaStream_t)stream);
    st.copy_in(b->d_latch, latch, sizeof(double) * 16 * N);
    st.copy_in(b->d_has, has, sizeof(int32_t) * N);
    st.copy_in(b->d_latch_u, latch_u, sizeof(double) * 16);
    st.copy_in(b->d_latch_u + 16, latch_u, sizeof(double) * 16);
    if (st.rc) return st.rc;
    if (has) b->imu_seen = true; // T9: a restored filter may carry a latched IMU sample
    b->stepped = true;
    return st.finish();
}

extern "C" int kfpos_batch_get_state(kfpos_batch *b, double *x, double *P, int32_t *status, void *stream) {
    if (!b || b->model == KFPOS_MODEL_ML) return KFPOS_ERR_INVALID;
    DeviceGuard g(b->device);
    cudaStream_t s = (cudaStream_t)stream;
    const size_t N = (size_t)b->N;
    Staging st(b, s);
    st.copy_out(x, b->d_x, sizeof(double) * b->n * N);
    double *d_P = st.out(P, sizeof(double) * b->n * b->n * N);
    if (st.rc) return st.rc;
    if (d_P) CK(launch_unpack_cov(b->n, b->N, b->d_P, d_P, s));
    st.copy_out(status, b->d_status, sizeof(int32_t) * N);
    return st.finish();
}

// ------------------------------------------------------------------- TOA steps
namespace {

// launches the T6 replay kernel over T steps whose ranges (and optional
// per-ranging errors) are already on the device
int launch_t6(kfpos_batch *b, int T, const double *d_dt, const void *d_ranges, int fmt,
              double err_scalar, const double *d_err, double *d_traj, int32_t *d_sel, cudaStream_t s,
              const double *d_dt_f = nullptr);
int run_events(kfpos_batch *b, Staging &st, int n, const kfpos_event *events, const void *d_ranges, int fmt,
               double err_scalar, const double *d_err, const double *d_sensors, double *d_traj, cudaStream_t s,
               const double *d_dt_f = nullptr);

} // namespace

extern "C" int kfpos_batch_replay_toa(kfpos_batch *b, int n_steps, const double *dt, const void *ranges,
                                      int fmt, double err_scalar, const double *err_var, double *traj,
                                      int32_t *sel, void *stream) {
    if (!b || b->model == KFPOS_MODEL_ML || n_steps < 0 || !dt || !ranges || !fmt_ok(fmt)) return KFPOS_ERR_INVALID;
    if (!b->have_anchors) return KFPOS_ERR_NOT_READY;
    if (n_steps == 0) return KFPOS_OK;
    if (es_check(b, n_steps)) return KFPOS_ERR_INVALID;
    if (sel && b->model != KFPOS_MODEL_T6) return KFPOS_ERR_INVALID; // leave-one-out exists only in T6
    DeviceGuard g(b->device);
    cudaStream_t s = (cudaStream_t)stream;
    const size_t N = (size_t)b->N, M = (size_t)b->anchors.n;
    const int T = n_steps;
    const size_t range_bytes = M * N * T * fmt_size(fmt), err_bytes = sizeof(double) * M * N * T;
    Staging st(b, s);
    double *d_traj = st.out(traj, sizeof(double) * 3 * N * T);
    int32_t *d_sel = st.out(sel, sizeof(int32_t) * N * T);
    int rc = KFPOS_OK;
    if (b->model != KFPOS_MODEL_T6) {
        // K8 / T9: a TOA-only schedule through the event-stream kernel
        std::vector<double> hdt(T);
        if ((rc = to_host(hdt.data(), dt, sizeof(double) * T))) return rc;
        const std::vector<kfpos_event> evs = toa_schedule(T, M, hdt.data());
        const void *d_r = st.in(ranges, range_bytes);
        const double *d_e = st.in(err_var, err_bytes);
        rc = run_events(b, st, T, evs.data(), d_r, fmt, err_scalar, d_e, nullptr, d_traj, s);
        return rc ? rc : st.finish();
    }
    const double *d_dt = st.ctl(dt, sizeof(double) * T); // small: always staged
    if (on_device(ranges) || err_var) {
        // the whole log on the device (host arrays staged whole)
        const void *d_r = st.in(ranges, range_bytes);
        const double *d_e = st.in(err_var, err_bytes);
        if (st.rc) return st.rc;
        rc = launch_t6(b, T, d_dt, d_r, fmt, err_scalar, d_e, d_traj, d_sel, s);
    } else {
        if (st.rc) return st.rc;
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
            rc = launch_t6(b, (int)tc, d_dt + t0, b->stage[k].p, fmt, err_scalar, nullptr,
                           d_traj ? d_traj + t0 * 3 * N : nullptr, d_sel ? d_sel + t0 * N : nullptr, s);
            if (rc) return rc;
            CK(cudaEventRecord(b->ev_done[k], s));
        }
        st.sync = true; // the host log is read by the chunk copies
    }
    return rc ? rc : st.finish();
}

extern "C" int kfpos_batch_replay_epochs(kfpos_batch *b, int n_steps, const double *dt_per_filter, const void *ranges,
                                         int fmt, double err_scalar, const double *err_var, double *traj,
                                         void *stream) {
    if (!b || n_steps < 0 || !dt_per_filter || !ranges) return KFPOS_ERR_INVALID;
    if (b->model != KFPOS_MODEL_T6 && b->model != KFPOS_MODEL_K8 && b->model != KFPOS_MODEL_T9) return KFPOS_ERR_INVALID;
    if (!fmt_ok(fmt)) return KFPOS_ERR_INVALID;
    if (!b->have_anchors) return KFPOS_ERR_NOT_READY;
    if (n_steps == 0) return KFPOS_OK;
    if (es_check(b, n_steps)) return KFPOS_ERR_INVALID;
    DeviceGuard g(b->device);
    cudaStream_t s = (cudaStream_t)stream;
    const size_t N = (size_t)b->N, M = (size_t)b->anchors.n, T = (size_t)n_steps;
    Staging st(b, s);
    const double *d_dtf = st.in(dt_per_filter, sizeof(double) * N * T);
    const void *d_r = st.in(ranges, M * N * T * fmt_size(fmt));
    const double *d_e = st.in(err_var, sizeof(double) * M * N * T);
    double *d_traj = st.out(traj, sizeof(double) * 3 * N * T);
    int rc;
    if (b->model == KFPOS_MODEL_T6) {
        if (st.rc) return st.rc;
        rc = launch_t6(b, n_steps, nullptr, d_r, fmt, err_scalar, d_e, d_traj, nullptr, s, d_dtf);
    } else { // K8 / T9: the epochs as a schedule of ranging events whose time steps are per filter
        const std::vector<kfpos_event> evs = toa_schedule(T, M, nullptr);
        rc = run_events(b, st, n_steps, evs.data(), d_r, fmt, err_scalar, d_e, nullptr, d_traj, s, d_dtf);
    }
    return rc ? rc : st.finish();
}

extern "C" int kfpos_batch_step_toa(kfpos_batch *b, double dt, const void *ranges, int fmt, double err_scalar,
                                    const double *err_var, void *stream) {
    return kfpos_batch_replay_toa(b, 1, &dt, ranges, fmt, err_scalar, err_var, nullptr, nullptr, stream);
}

namespace {

int launch_t6(kfpos_batch *b, int T, const double *d_dt, const void *d_ranges, int fmt,
              double err_scalar, const double *d_err, double *d_traj, int32_t *d_sel, cudaStream_t s,
              const double *d_dt_f) {
    b->stepped = true;
    T6Params p;
    if (int rc = bind_replay(b, p, make_rs(b, d_ranges, fmt, err_scalar, d_err), d_dt_f, d_traj, T, s)) return rc;
    p.T = T;
    p.ignore_worst = b->cfg.ignore_worst_anchor;
    p.variant = b->cfg.variant;
    p.n_ignore = b->cfg.num_ignored_rangings;
    p.best_mode = b->cfg.best_mode;
    p.ignore_thr = b->cfg.ignore_cost_threshold;
    p.accel_noise = b->cfg.accel_noise;
    p.dt = d_dt;
    p.sel = d_sel;
    CK(launch_t6_replay(p, s));
    return replayed(b, s);
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

// events: HOST array, staged through `st`; every data pointer already on the device.  The caller's staging errors
// are returned before anything is launched.
int run_events(kfpos_batch *b, Staging &st, int n, const kfpos_event *events, const void *d_ranges, int fmt,
               double err_scalar, const double *d_err, const double *d_sensors, double *d_traj, cudaStream_t s,
               const double *d_dt_f) {
    static_assert(sizeof(kfpos_event) == sizeof(EventDesc), "kfpos_event and EventDesc must have one layout");
    if (st.rc) return st.rc;
    if (n <= 0) return KFPOS_OK;
    b->stepped = true;
    const EventDesc *d_events = st.ctl((const EventDesc *)events, sizeof(EventDesc) * (size_t)n);
    if (st.rc) return st.rc;
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
        if (int rc = bind_replay(b, p, rs, d_dt_f, d_traj, n_toa, s)) return rc;
        p.cfg = make_k8cfg(b);
        p.sensors = d_sensors;
        p.events = d_events;
        p.n_events = n;
        p.latch = b->d_latch;
        p.has = b->d_has;
        p.latch_u = b->d_latch_u;
        p.uninit = track_uninit ? b->d_uninit : nullptr;
        CK(launch_k8_replay(p, s));
        break;
    }
    case KFPOS_MODEL_T9: {
        T9Params p;
        if (int rc = bind_replay(b, p, rs, d_dt_f, d_traj, n_toa, s)) return rc;
        p.accel_noise = b->cfg.accel_noise;
        p.jolt = b->cfg.jolt;
        p.sensors = d_sensors;
        p.events = d_events;
        p.n_events = n;
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
        CK(launch_t9_replay(p, s));
        break;
    }
    default: return KFPOS_ERR_INVALID;
    }
    int rc = replayed(b, s);
    if (!rc && track_uninit) rc = fetch_uninit(b, s);
    return rc;
}

} // namespace

static int replay_events_impl(kfpos_batch *b, int n_events, const kfpos_event *events, const double *dt_per_filter,
                              const void *ranges, int fmt, double err_scalar, const double *err_var,
                              const double *sensors, int64_t sensor_rows, double *traj, void *stream) {
    if (!b || (b->model != KFPOS_MODEL_K8 && b->model != KFPOS_MODEL_T9) || n_events < 0 || !events)
        return KFPOS_ERR_INVALID;
    if (!fmt_ok(fmt)) return KFPOS_ERR_INVALID;
    if (!b->have_anchors) return KFPOS_ERR_NOT_READY;
    if (n_events == 0) return KFPOS_OK;
    DeviceGuard g(b->device);
    cudaStream_t s = (cudaStream_t)stream;
    const size_t N = (size_t)b->N, M = (size_t)b->anchors.n;
    int64_t range_rows = 0, n_toa = 0;
    for (int e = 0; e < n_events; ++e) {
        const kfpos_event &ev = events[e];
        const int rows = event_rows(ev.kind, (int)M);
        if (rows < 0 || ev.offset < 0) return KFPOS_ERR_INVALID;
        if (b->model == KFPOS_MODEL_T9 && ev.kind != KFPOS_EV_TOA && ev.kind != KFPOS_EV_IMU) return KFPOS_ERR_INVALID;
        if (ev.kind == KFPOS_EV_TOA) {
            if (!ranges) return KFPOS_ERR_INVALID;
            if (ev.offset + rows > range_rows) range_rows = ev.offset + rows;
            ++n_toa;
        } else {
            if (!sensors || ev.offset + rows > sensor_rows) return KFPOS_ERR_INVALID;
        }
    }
    if (es_check(b, n_toa)) return KFPOS_ERR_INVALID;
    Staging st(b, s);
    const void *d_r = st.in(ranges, (size_t)range_rows * N * fmt_size(fmt));
    const double *d_e = st.in(err_var, sizeof(double) * (size_t)range_rows * N);
    const double *d_s = st.in(sensors, sizeof(double) * (size_t)sensor_rows * N);
    double *d_traj = st.out(traj, sizeof(double) * 3 * N * (size_t)n_toa);
    const double *d_dtf = st.in(dt_per_filter, sizeof(double) * N * (size_t)n_events);
    int rc = run_events(b, st, n_events, events, d_r, fmt, err_scalar, d_e, d_s, d_traj, s, d_dtf);
    return rc ? rc : st.finish();
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

// one non-TOA event whose payload rows are gathered into one device array
int single_sensor_event(kfpos_batch *b, Staging &st, int kind, double dt, const double *const *rows, int n_rows,
                        const double aux[9], cudaStream_t s) {
    const size_t N = (size_t)b->N;
    double *dst = st.buf<double>(sizeof(double) * N * (size_t)n_rows);
    if (st.rc) return st.rc;
    for (int i = 0; i < n_rows; ++i) {
        if (!rows[i]) return KFPOS_ERR_INVALID;
        st.copy_in(dst + (size_t)i * N, rows[i], sizeof(double) * N);
    }
    kfpos_event ev;
    memset(&ev, 0, sizeof ev);
    ev.kind = kind;
    ev.dt = dt;
    ev.offset = 0;
    if (aux) memcpy(ev.aux, aux, sizeof ev.aux);
    int rc = run_events(b, st, 1, &ev, nullptr, KFPOS_FMT_F64_M, 1.0, nullptr, dst, nullptr, s);
    return rc ? rc : st.finish();
}

} // namespace

extern "C" int kfpos_batch_step_px4(kfpos_batch *b, double dt, const double *integration_x,
                                    const double *integration_y, const double *integration_rot_z,
                                    const double *integration_time_us, const int32_t *quality, void *stream) {
    if (!b || b->model != KFPOS_MODEL_K8 || !quality) return KFPOS_ERR_INVALID;
    DeviceGuard g(b->device);
    cudaStream_t s = (cudaStream_t)stream;
    const size_t N = (size_t)b->N;
    Staging st(b, s);
    const int32_t *d_q = st.in(quality, sizeof(int32_t) * N);
    double *d_qf = st.buf<double>(sizeof(double) * N);
    if (st.rc) return st.rc;
    CK(launch_i32_to_f64(b->N, d_q, d_qf, s));
    const double *rows[5] = {integration_x, integration_y, integration_rot_z, integration_time_us, d_qf};
    return single_sensor_event(b, st, KFPOS_EV_PX4, dt, rows, 5, nullptr, s);
}

extern "C" int kfpos_batch_step_imu(kfpos_batch *b, double dt, const double *ang_vel, const double *cov_ang_vel,
                                    const double *lin_acc, const double *cov_acc, void *stream) {
    if (!b || (b->model != KFPOS_MODEL_K8 && b->model != KFPOS_MODEL_T9) || !lin_acc) return KFPOS_ERR_INVALID;
    DeviceGuard g(b->device);
    cudaStream_t s = (cudaStream_t)stream;
    const size_t N = (size_t)b->N;
    Staging st(b, s);
    double aux[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
    if (b->model == KFPOS_MODEL_K8) {
        if (!ang_vel) return KFPOS_ERR_INVALID;
        if (cov_acc) { aux[0] = cov_acc[0]; aux[1] = cov_acc[1]; aux[2] = cov_acc[3]; aux[3] = cov_acc[4]; }
        if (cov_ang_vel) aux[4] = cov_ang_vel[8];
        const double *rows[3] = {ang_vel + 2 * N, lin_acc, lin_acc + N};
        return single_sensor_event(b, st, KFPOS_EV_IMU, dt, rows, 3, aux, s);
    }
    if (cov_acc) memcpy(aux, cov_acc, sizeof aux);
    const double *rows[3] = {lin_acc, lin_acc + N, lin_acc + 2 * N};
    return single_sensor_event(b, st, KFPOS_EV_IMU, dt, rows, 3, aux, s);
}

extern "C" int kfpos_batch_step_mag(kfpos_batch *b, double dt, const double *mag, void *stream) {
    if (!b || b->model != KFPOS_MODEL_K8 || !mag) return KFPOS_ERR_INVALID;
    DeviceGuard g(b->device);
    Staging st(b, (cudaStream_t)stream);
    const double *rows[2] = {mag, mag + (size_t)b->N};
    return single_sensor_event(b, st, KFPOS_EV_MAG, dt, rows, 2, nullptr, (cudaStream_t)stream);
}

extern "C" int kfpos_batch_step_compass(kfpos_batch *b, double dt, const double *compass, void *stream) {
    if (!b || b->model != KFPOS_MODEL_K8 || !compass) return KFPOS_ERR_INVALID;
    DeviceGuard g(b->device);
    Staging st(b, (cudaStream_t)stream);
    const double *rows[1] = {compass};
    return single_sensor_event(b, st, KFPOS_EV_COMPASS, dt, rows, 1, nullptr, (cudaStream_t)stream);
}

// --------------------------------------------------------------------- getPose
namespace {
// the model's getPose prediction into the device arrays dx (SoA [n][N]) and dP (SoA [n][n][N])
int enqueue_get_pose(kfpos_batch *b, double dt, double *dx, double *dP, cudaStream_t s) {
    switch (b->model) {
    case KFPOS_MODEL_T6: CK(launch_t6_get_pose(b->N, dt, b->cfg.accel_noise, b->d_x, b->d_P, dx, dP, s)); break;
    case KFPOS_MODEL_K8:
        CK(launch_k8_get_pose(b->N, dt, b->cfg.accel_noise, b->cfg.jolt, b->d_x, b->d_P, dx, dP, s));
        break;
    case KFPOS_MODEL_T9: CK(launch_t9_get_pose(b->N, dt, b->cfg.jolt, b->d_x, b->d_P, dx, dP, s)); break;
    default: return KFPOS_ERR_UNSUPPORTED;
    }
    return KFPOS_OK;
}
} // namespace

extern "C" int kfpos_batch_get_pose(kfpos_batch *b, double dt, double *x_pred, double *P_pred, void *stream) {
    if (!b || b->model == KFPOS_MODEL_ML) return KFPOS_ERR_INVALID;
    DeviceGuard g(b->device);
    cudaStream_t s = (cudaStream_t)stream;
    const size_t N = (size_t)b->N;
    Staging st(b, s);
    double *dx = st.out(x_pred, sizeof(double) * b->n * N);
    double *dP = st.out(P_pred, sizeof(double) * b->n * b->n * N);
    if (st.rc) return st.rc;
    int rc = enqueue_get_pose(b, dt, dx, dP, s);
    return rc ? rc : st.finish();
}

extern "C" int kfpos_batch_get_pose_msg(kfpos_batch *b, double dt, double *pose13, double *cov36, void *stream) {
    if (!b || b->model == KFPOS_MODEL_ML) return KFPOS_ERR_INVALID;
    if (!b->stepped) return KFPOS_ERR_NOT_READY; // getPose returns false before the first measurement
    DeviceGuard g(b->device);
    cudaStream_t s = (cudaStream_t)stream;
    const size_t N = (size_t)b->N;
    Staging st(b, s);
    double *dx = st.buf<double>(sizeof(double) * b->n * N);
    double *dP = st.buf<double>(sizeof(double) * b->n * b->n * N);
    double *d_pose = st.out(pose13, sizeof(double) * 13 * N);
    double *d_cov = st.out(cov36, sizeof(double) * 36 * N);
    if (st.rc) return st.rc;
    int rc = enqueue_get_pose(b, dt, dx, dP, s);
    if (rc) return rc;
    const int model = b->model == KFPOS_MODEL_T6 ? 1 : (b->model == KFPOS_MODEL_K8 ? 2 : 3);
    // K8 without useFixedHeight: the tag height of an ML-initialised filter is its own (KF.cpp:256-257, 328-332)
    const double *tagz = (b->model == KFPOS_MODEL_K8 && b->cfg.ml_initial_position && !b->cfg.use_fixed_height)
                             ? b->d_latch + 9 * N : nullptr;
    CK(launch_pose_msg(model, b->N, b->cfg.fixed_height, tagz, dx, dP, d_pose, d_cov, s));
    return st.finish();
}

// -------------------------------------------------------------------------- ML
extern "C" int kfpos_batch_ml_solve(kfpos_batch *b, const void *ranges, int fmt, double err_scalar,
                                    const double *err_var, double *pos, double *cov, int32_t *iters,
                                    int32_t *sel, int32_t *status, void *stream) {
    if (!b || b->model != KFPOS_MODEL_ML || !ranges || !fmt_ok(fmt)) return KFPOS_ERR_INVALID;
    if (!b->have_anchors) return KFPOS_ERR_NOT_READY;
    DeviceGuard g(b->device);
    cudaStream_t s = (cudaStream_t)stream;
    const size_t N = (size_t)b->N, M = (size_t)b->anchors.n;
    Staging st(b, s);
    const void *d_r = st.in(ranges, M * N * fmt_size(fmt));
    const double *d_e = st.in(err_var, sizeof(double) * M * N);
    MlParams p;
    p.anchors = b->anchors;
    p.rs = make_rs(b, d_r, fmt, err_scalar, d_e);
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
    p.pos = st.out(pos, sizeof(double) * 3 * N);
    p.cov = st.out(cov, sizeof(double) * 9 * N);
    p.iters = st.out(iters, sizeof(int32_t) * N);
    p.sel = st.out(sel, sizeof(int32_t) * 2 * N);
    p.status = st.out(status, sizeof(int32_t) * N);
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
        p.xw_scratch = st.buf(bytes);
        p.xw_scratch_bytes = bytes;
    }
    if (st.rc) return st.rc;
    CK(launch_ml_solve(p, s));
    return st.finish();
}

// ------------------------------------------------------------ epoch assembler
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
    if (int rc = check_device(device)) return rc;
    DeviceGuard g(device);
    if (!g.ok) return KFPOS_ERR_CUDA;
    cudaStream_t s = (cudaStream_t)stream;
    const size_t N = (size_t)n_logs, L = (size_t)n_msgs, M = (size_t)n_anchors, T = (size_t)max_epochs;
    Staging st(s);
    AssembleParams p;
    p.anchor = st.in(anchor, L * N); p.seq = st.in(seq, L * N);
    p.range_mm = st.in(range_mm, 4 * L * N); p.err = st.in(err, 8 * L * N); p.t = st.in(t, 8 * L * N);
    p.ranges_out = st.out(ranges_out, 4 * T * M * N); p.err_out = st.out(err_out, 8 * T * M * N);
    p.dt_out = st.out(dt_out, 8 * T * N);
    p.n_epochs = st.out(n_epochs, 4 * N);
    p.t_out = st.out(t_out, 8 * T * N);
    if (st.rc) return st.rc;
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
    p.N = n_logs; p.L = n_msgs; p.max_epochs = max_epochs;
    p.M = n_anchors; p.fix_b12 = fix; p.first_dt = first_dt;
    p.tbl_r = (int32_t *)tr.p; p.tbl_e = (double *)te.p;
    CK(launch_assemble(p, s));
    // With device pointers only, the call is asynchronous on `stream` like the rest of the API (the table
    // is reused by the next call on the same device, which is ordered behind this one only if it
    // uses the same stream: callers on different streams must synchronise themselves).
    return st.finish();
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
    int64_t range_rows = 0, sensor_rows = 0;
    std::vector<int64_t> slot_row((size_t)n_slots);
    for (int sidx = 0; sidx < n_slots; ++sidx) {
        const int k = slot_kind[sidx];
        const int rows = event_rows(k, n_anchors);
        if (rows < 0) return KFPOS_ERR_INVALID;
        int64_t &used = k == KFPOS_EV_TOA ? range_rows : sensor_rows;
        slot_row[sidx] = used;
        used += rows;
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
    if (int rc = check_device(device)) return rc;
    DeviceGuard g(device);
    if (!g.ok) return KFPOS_ERR_CUDA;
    cudaStream_t s = (cudaStream_t)stream;
    const size_t N = (size_t)n_logs, M = (size_t)n_anchors;
    const size_t range_n = (size_t)(range_rows > 0 ? range_rows : 1) * N;
    const size_t sensor_n = (size_t)(sensor_rows > 0 ? sensor_rows : 1) * N;
    Staging st(s); // the slot tables are always staged, so the call always synchronises
    MergeParams p;
    memset(&p, 0, sizeof p);
    p.N = n_logs; p.M = n_anchors; p.n_slots = n_slots; p.first_dt = first_dt;
    p.L[0] = n_epochs;
    p.t_src[0] = st.in(t_epoch, 8 * (size_t)n_epochs * N);
    p.ranges = st.in(ranges, 4 * (size_t)n_epochs * M * N);
    p.err_src = st.in(err, 8 * (size_t)n_epochs * M * N);
    for (int k = 1; k < 5; ++k) {
        const int64_t Lk = n_samples ? n_samples[k - 1] : 0;
        if (Lk <= 0 || !t_sensor || !payload || !t_sensor[k - 1] || !payload[k - 1]) continue;
        p.L[k] = Lk;
        p.t_src[k] = st.in(t_sensor[k - 1], 8 * (size_t)Lk * N);
        p.src[k] = st.in(payload[k - 1], 8 * (size_t)Lk * event_rows(k, n_anchors) * N);
    }
    p.slot_kind = st.ctl(slot_kind, sizeof(int32_t) * (size_t)n_slots);
    p.slot_row = st.ctl(slot_row.data(), sizeof(int64_t) * (size_t)n_slots);
    p.dt_f = st.out(dt_out, 8 * (size_t)n_slots * N);
    p.ranges_out = st.out(ranges_out, 4 * range_n);
    p.err_out = st.out(err_out, 8 * range_n);
    p.sensors_out = st.out(sensors_out, 8 * sensor_n);
    p.n_dropped = st.out(n_dropped, 4 * N);
    if (st.rc) return st.rc;
    // slots nobody takes keep "no ranging" / zero payloads
    if (p.ranges_out) CK(cudaMemsetAsync(p.ranges_out, 0xff, 4 * range_n, s));
    if (p.err_out) CK(cudaMemsetAsync(p.err_out, 0, 8 * range_n, s));
    if (p.sensors_out) CK(cudaMemsetAsync(p.sensors_out, 0, 8 * sensor_n, s));
    CK(launch_merge(p, s));
    return st.finish();
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
int enqueue_error_stats(kfpos_batch *b, Staging &st, const double *truth, cudaStream_t s) {
    const double *d_truth = nullptr;
    if (truth) {
        d_truth = st.in(truth, sizeof(double) * 3 * (size_t)b->N);
        if (st.rc) return st.rc;
    } else if (!b->partials_fresh) {
        if (!b->d_truth) return KFPOS_ERR_NOT_READY;
        d_truth = b->d_truth; // registered, but the state changed since the last replay (single steps, set_state)
    }
    // K8 is planar: z is the configured tag height (KF.cpp:328-332)
    CK(launch_error_stats(b->N, b->d_x, b->model == KFPOS_MODEL_K8 ? -1 : 2, b->cfg.fixed_height, b->d_status,
                          d_truth, b->d_partials, b->d_out4, s));
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

// ONE collective: the `count` 8-byte values at `send` of every rank to every rank, [rank][count] in `recv` (grown
// to fit); the number of ranks comes back in `n_ranks`
constexpr int NCCL_UINT64 = 5, NCCL_DOUBLE = 8; // ncclDataType_t
int all_gather(struct ncclComm *comm, const void *send, size_t count, DevBuf &recv, int *n_ranks, cudaStream_t s,
               int type = NCCL_DOUBLE) {
    NcclApi &api = nccl_api();
    if (!api.all_gather || !api.count) return KFPOS_ERR_UNSUPPORTED;
    if (api.count(comm, n_ranks) != 0 || *n_ranks < 1 || *n_ranks > 1024) return KFPOS_ERR_INVALID;
    CK(recv.reserve(sizeof(double) * count * (size_t)*n_ranks));
    return api.all_gather(send, recv.p, count, type, comm, s) != 0 ? KFPOS_ERR_CUDA : KFPOS_OK;
}
} // namespace

extern "C" int kfpos_batch_error_stats(kfpos_batch *b, const double *truth, double out[4], void *stream) {
    if (!b || b->model == KFPOS_MODEL_ML) return KFPOS_ERR_INVALID;
    DeviceGuard g(b->device);
    cudaStream_t s = (cudaStream_t)stream;
    Staging st(b, s);
    int rc = enqueue_error_stats(b, st, truth, s);
    if (rc) return rc;
    st.copy_out(out, b->d_out4, sizeof(double) * 4); // out == null: the result stays on the device (allreduce)
    return st.finish();
}

extern "C" int kfpos_stats_allreduce(kfpos_batch *b, struct ncclComm *comm, const double *truth, double out[6],
                                     void *stream) {
    if (!b || b->model == KFPOS_MODEL_ML || !out) return KFPOS_ERR_INVALID;
    DeviceGuard g(b->device);
    cudaStream_t s = (cudaStream_t)stream;
    Staging st(b, s);
    int rc;
    // truth == null: what the last kfpos_batch_error_stats left on the device, if the state has not changed since
    if ((truth || !b->out4_valid) && (rc = enqueue_error_stats(b, st, truth, s))) return rc;
    const double *d_res = b->d_out4;
    if (comm) {
        // every rank's 4 doubles to every rank, then the same pairwise tree over the rank index on every rank --
        // the top levels of the global tree, in a fixed order
        int n_ranks = 0;
        if ((rc = all_gather(comm, b->d_out4, 4, b->gather, &n_ranks, s))) return rc;
        double *gat = (double *)b->gather.p;
        CK(launch_error_stats_tree(n_ranks, gat, gat, s));
        d_res = gat;
    }
    st.copy_out(out, d_res, sizeof(double) * 4);
    if ((rc = st.finish())) return rc;
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
    cudaFree(b->d_eh_counts);
    b->d_etruth_own = b->d_escratch = b->d_efold = b->d_eout = nullptr;
    b->d_eh_counts = nullptr;
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
    // a registered histogram gets its counts with the rows (kfpos_batch_set_error_hist)
    const size_t hbytes = sizeof(unsigned long long) * (size_t)b->eh_bins * (size_t)n_rows;
    if (e == cudaSuccess && hbytes) e = cudaMalloc((void **)&b->d_eh_counts, hbytes);
    if (e == cudaSuccess && hbytes) e = cudaMemsetAsync(b->d_eh_counts, 0, hbytes, s);
    const size_t tbytes = sizeof(double) * 3 * (size_t)b->N * (size_t)n_rows;
    if (e == cudaSuccess && !dev) e = cudaMalloc((void **)&b->d_etruth_own, tbytes);
    if (e == cudaSuccess && !dev) e = cudaMemcpyAsync(b->d_etruth_own, truth, tbytes, cudaMemcpyHostToDevice, s);
    if (e == cudaSuccess && !dev) e = cudaStreamSynchronize(s);
    if (e != cudaSuccess) {
        cudaFree(b->d_etruth_own);
        cudaFree(b->d_escratch);
        cudaFree(b->d_efold);
        cudaFree(b->d_eout);
        cudaFree(b->d_eh_counts);
        b->d_etruth_own = b->d_escratch = b->d_efold = b->d_eout = nullptr;
        b->d_eh_counts = nullptr;
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
    Staging st(b, s);
    double *d_out = st.out(out, sizeof(double) * ES_W * (size_t)n_rows);
    if (st.rc) return st.rc;
    if ((rc = enqueue_epoch_stats(b, d_out, s))) return rc;
    return st.finish();
}

extern "C" int kfpos_epoch_stats_allreduce(kfpos_batch *b, struct ncclComm *comm, int64_t n_rows, double *out,
                                           void *stream) {
    int rc = es_ready(b, n_rows, out);
    if (rc) return rc;
    DeviceGuard g(b->device);
    cudaStream_t s = (cudaStream_t)stream;
    if ((rc = enqueue_epoch_stats(b, b->d_eout, s))) return rc;
    const double *d_res = b->d_eout;
    if (comm) {
        // every rank's [n_rows][6] to every rank ([rank][row][6]), then per row the pairwise tree over the rank
        // index -- the top levels of the global tree; row r's result lands on its rank-0 entry
        int n_ranks = 0;
        if ((rc = all_gather(comm, b->d_eout, (size_t)n_rows * ES_W, b->es_gather, &n_ranks, s))) return rc;
        double *gat = (double *)b->es_gather.p;
        CK(launch_stats_tree(ES_W, n_rows, n_ranks, gat, gat, ES_W, n_rows * ES_W, gat, s));
        d_res = gat;
    }
    Staging st(b, s);
    st.copy_out(out, d_res, sizeof(double) * ES_W * (size_t)n_rows);
    return st.finish();
}

// ------------------------------------------------------- per-epoch error histograms
extern "C" int kfpos_batch_set_error_hist(kfpos_batch *b, int quantity, int n_edges, const double *edges) {
    if (!b || b->model == KFPOS_MODEL_ML || n_edges < 0) return KFPOS_ERR_INVALID;
    const bool reg = n_edges > 0 && edges;
    std::vector<double> tbl(reg ? n_edges : 0);  // the caller's edges, then the device table
    if (reg) {
        if (quantity < KFPOS_HIST_ERR || quantity > KFPOS_HIST_NEES || n_edges > EH_MAX_BINS - 1) return KFPOS_ERR_INVALID;
        int rc = to_host(tbl.data(), edges, sizeof(double) * (size_t)n_edges);
        if (rc) return rc;
        const bool metres = quantity != KFPOS_HIST_NEES;
        for (int i = 0; i < n_edges; ++i) {
            const double v = tbl[i];
            if (!std::isfinite(v) || (metres && v < 0.0) || (i > 0 && !(v > tbl[i - 1]))) return KFPOS_ERR_INVALID;
        }
        // the error quantities are binned as e^2: the edges are squared here, once, so no kernel takes a root
        if (metres)
            for (double &v : tbl) v = v * v;
        tbl.resize(EH_MAX_BINS - 1, INFINITY); // the kernel's search always spans EH_MAX_BINS - 1 entries
    }
    DeviceGuard g(b->device);
    // (cudaFree waits for the device: no launch still reads the previous table or counts)
    cudaFree(b->d_eh_edges);
    cudaFree(b->d_eh_counts);
    b->d_eh_edges = nullptr;
    b->d_eh_counts = nullptr;
    b->eh_bins = b->eh_quantity = 0;
    if (!reg) return KFPOS_OK;
    const size_t hbytes = sizeof(unsigned long long) * (size_t)(n_edges + 1) * (size_t)b->es_rows;
    cudaError_t e = cudaMalloc((void **)&b->d_eh_edges, sizeof(double) * tbl.size());
    if (e == cudaSuccess) e = cudaMemcpy(b->d_eh_edges, tbl.data(), sizeof(double) * tbl.size(), cudaMemcpyHostToDevice);
    if (e == cudaSuccess && hbytes) e = cudaMalloc((void **)&b->d_eh_counts, hbytes);
    if (e == cudaSuccess && hbytes) e = cudaMemset(b->d_eh_counts, 0, hbytes);
    if (e != cudaSuccess) {
        cudaFree(b->d_eh_edges);
        cudaFree(b->d_eh_counts);
        b->d_eh_edges = nullptr;
        b->d_eh_counts = nullptr;
        cudaGetLastError();
        return map_cuda_err(e);
    }
    b->eh_quantity = quantity;
    b->eh_bins = n_edges + 1;
    return KFPOS_OK;
}

namespace {
int eh_ready(const kfpos_batch *b, int64_t n_rows, const uint64_t *counts) {
    if (!b || b->model == KFPOS_MODEL_ML || !counts) return KFPOS_ERR_INVALID;
    if (!b->d_eh_counts) return KFPOS_ERR_NOT_READY; // no histogram or no truth trajectory
    return n_rows == b->es_rows ? KFPOS_OK : KFPOS_ERR_INVALID;
}
// [es_rows][eh_bins] of this batch into the device array `d_out`: the rows the cursor has passed, the rest zero
int enqueue_error_hist(kfpos_batch *b, unsigned long long *d_out, cudaStream_t s) {
    const int64_t done = b->es_cursor < b->es_rows ? b->es_cursor : b->es_rows;
    const size_t row_bytes = sizeof(unsigned long long) * (size_t)b->eh_bins;
    if (done > 0) CK(cudaMemcpyAsync(d_out, b->d_eh_counts, row_bytes * (size_t)done, cudaMemcpyDeviceToDevice, s));
    if (done < b->es_rows) CK(cudaMemsetAsync(d_out + done * b->eh_bins, 0, row_bytes * (size_t)(b->es_rows - done), s));
    return KFPOS_OK;
}
} // namespace

extern "C" int kfpos_batch_error_hist(kfpos_batch *b, int64_t n_rows, uint64_t *counts, void *stream) {
    int rc = eh_ready(b, n_rows, counts);
    if (rc) return rc;
    DeviceGuard g(b->device);
    cudaStream_t s = (cudaStream_t)stream;
    Staging st(b, s);
    auto *d_out = (unsigned long long *)st.out(counts, sizeof(uint64_t) * (size_t)b->eh_bins * (size_t)n_rows);
    if (st.rc) return st.rc;
    if ((rc = enqueue_error_hist(b, d_out, s))) return rc;
    return st.finish();
}

extern "C" int kfpos_error_hist_allreduce(kfpos_batch *b, struct ncclComm *comm, int64_t n_rows, uint64_t *counts,
                                          void *stream) {
    int rc = eh_ready(b, n_rows, counts);
    if (rc) return rc;
    DeviceGuard g(b->device);
    cudaStream_t s = (cudaStream_t)stream;
    const size_t n = (size_t)b->eh_bins * (size_t)n_rows;
    Staging st(b, s);
    auto *d_out = (unsigned long long *)st.out(counts, sizeof(uint64_t) * n);
    if (st.rc) return st.rc;
    if (!comm) {
        if ((rc = enqueue_error_hist(b, d_out, s))) return rc;
        return st.finish();
    }
    // every rank's counts to every rank ([rank][row][bin]), then the integer sum over the rank index: exact in
    // any order, so any split of the filters over the ranks gives the single-GPU counts
    unsigned long long *d_mine = st.buf<unsigned long long>(sizeof(uint64_t) * n);
    if (st.rc) return st.rc;
    if ((rc = enqueue_error_hist(b, d_mine, s))) return rc;
    int n_ranks = 0;
    if ((rc = all_gather(comm, d_mine, n, b->eh_gather, &n_ranks, s, NCCL_UINT64))) return rc;
    CK(launch_sum_ranks_u64(n_ranks, (int64_t)n, (const unsigned long long *)b->eh_gather.p, d_out, s));
    return st.finish();
}

extern "C" int kfpos_measure_fp64_peak(int device, double *flops_per_s) {
    if (!flops_per_s) return KFPOS_ERR_INVALID;
    if (int rc = check_device(device)) return rc;
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
    for (int i = 0; i < n_events; ++i) { // every event must write inside the tensors it was given (no MAG samples)
        const int rows = events[i].kind == KFPOS_EV_MAG ? -1 : event_rows(events[i].kind, n_anchors);
        const int64_t lim = events[i].kind == KFPOS_EV_TOA ? range_rows : sensor_rows;
        if (rows < 0 || events[i].offset < 0 || events[i].offset + rows > lim) return KFPOS_ERR_INVALID;
        if ((events[i].kind == KFPOS_EV_TOA && !ranges) || (events[i].kind != KFPOS_EV_TOA && !sensors))
            return KFPOS_ERR_INVALID;
    }
    if (int rc = check_device(device)) return rc;
    DeviceGuard g(device);
    if (!g.ok) return KFPOS_ERR_CUDA;
    cudaStream_t s = (cudaStream_t)stream;
    const size_t N = (size_t)n_filters;
    SynthK8Params p;
    int rc = anchor_table(n_anchors, anchors_xyz, &p.anchors);
    if (rc) return rc;
    Staging st(s);
    p.ranges = st.out(ranges, 4 * (size_t)range_rows * N);
    p.sensors = st.out(sensors, 8 * (size_t)sensor_rows * N);
    p.x0 = st.out(x0, 8 * 8 * N);
    p.truth_end = st.out(truth_end, 8 * 3 * N);
    if (st.rc) return st.rc;
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
            CK(cudaDeviceSynchronize()); // growing a slot frees the old one: nothing may still read it
            CK(slot.reserve(sizeof(SynthEvent) * (size_t)(n_events < 256 ? 256 : n_events)));
        }
        d_ev = slot.p;
        CK(cudaMemcpyAsync(d_ev, events, sizeof(SynthEvent) * (size_t)n_events, cudaMemcpyHostToDevice, s));
    }
    p.N = n_filters; p.filter0 = first_filter; p.seed = seed; p.M = n_anchors; p.n_events = n_events;
    p.tag_z = tag_z; p.sigma_r = sigma_r; p.t_end = t_end;
    p.events = (const SynthEvent *)d_ev;
    CK(launch_synth_k8(p, s));
    return st.finish();
}

extern "C" int kfpos_synth_k8_truth(int device, int64_t n_filters, int64_t first_filter, uint64_t seed, int n_times,
                                    const double *t, double tag_z, double *truth, void *stream) {
    if (n_filters <= 0 || n_times < 0 || (n_times > 0 && (!t || !truth))) return KFPOS_ERR_INVALID;
    if (int rc = check_device(device)) return rc;
    if (n_times == 0) return KFPOS_OK;
    DeviceGuard g(device);
    if (!g.ok) return KFPOS_ERR_CUDA;
    cudaStream_t s = (cudaStream_t)stream;
    Staging st(s);
    SynthTruthParams p;
    p.N = n_filters; p.filter0 = first_filter; p.seed = seed; p.n_times = n_times; p.tag_z = tag_z;
    p.t = st.in(t, sizeof(double) * (size_t)n_times);
    p.truth = st.out(truth, sizeof(double) * 3 * (size_t)n_filters * (size_t)n_times);
    if (st.rc) return st.rc;
    CK(launch_synth_k8_truth(p, s));
    return st.finish();
}

namespace {
// kfpos_synth_toa_ranges with an optional NLOS mask output (kfpos_synth_toa_ranges_nlos)
int synth_toa_ranges(int device, int64_t n_filters, int n_anchors, const double *anchors_xyz, int n_epochs,
                     const double *t, const kfpos_synth_toa *gen, int fmt, void *ranges, uint32_t *nlos, void *stream) {
    const auto prob = [](double q) { return q >= 0.0 && q <= 1.0; }; // false for NaN
    if (n_filters <= 0 || n_anchors <= 0 || n_anchors > KFPOS_MAX_ANCHORS || !anchors_xyz || n_epochs < 0 ||
        (n_epochs > 0 && (!t || !ranges)) || !gen || (fmt != KFPOS_FMT_I32_MM && fmt != KFPOS_FMT_U16_MM))
        return KFPOS_ERR_INVALID;
    if (!prob(gen->p_missing) || !prob(gen->p_nlos) || !(gen->sigma_r >= 0.0) ||
        (gen->p_nlos > 0.0 && !(gen->nlos_mean > 0.0)) || gen->first_filter < 0 || gen->first_epoch < 0 ||
        gen->first_epoch + n_epochs > (int64_t)0xFFFFFFFF) // epoch index 0xFFFFFFFF: the per-filter constants
        return KFPOS_ERR_INVALID;
    if (int rc = check_device(device)) return rc;
    if (n_epochs == 0) return KFPOS_OK;
    DeviceGuard g(device);
    if (!g.ok) return KFPOS_ERR_CUDA;
    cudaStream_t s = (cudaStream_t)stream;
    const size_t row = fmt_size(fmt) * (size_t)n_anchors * (size_t)n_filters; // bytes of one epoch
    const size_t mask_row = sizeof(uint32_t) * (size_t)n_filters;
    // the epoch times travel in the parameter block, SYNTH_TOA_T per launch: nothing to stage, so device outputs
    // leave the call asynchronous (the next chunk can be generated while this one is replayed)
    SynthToaParams p{};
    int rc = anchor_table(n_anchors, anchors_xyz, &p.anchors);
    if (rc) return rc;
    Staging st(s);
    char *d_r = st.out((char *)ranges, row * (size_t)n_epochs);
    uint32_t *d_m = st.out(nlos, mask_row * (size_t)n_epochs);
    if (st.rc) return st.rc;
    p.N = n_filters; p.filter0 = gen->first_filter; p.seed = gen->seed; p.M = n_anchors;
    p.tag_z = gen->tag_z; p.sigma_r = gen->sigma_r; p.p_missing = gen->p_missing; p.p_nlos = gen->p_nlos;
    p.nlos_mean = gen->nlos_mean;
    for (int k0 = 0; k0 < n_epochs; k0 += SYNTH_TOA_T) {
        p.n_epochs = n_epochs - k0 < SYNTH_TOA_T ? n_epochs - k0 : SYNTH_TOA_T;
        p.epoch0 = (uint32_t)(gen->first_epoch + k0);
        memcpy(p.t, t + k0, sizeof(double) * (size_t)p.n_epochs);
        p.ranges = d_r + row * (size_t)k0;
        p.nlos = d_m ? d_m + (size_t)n_filters * (size_t)k0 : nullptr;
        CK(launch_synth_toa(p, fmt == KFPOS_FMT_U16_MM, s));
    }
    return st.finish();
}
} // namespace

extern "C" int kfpos_synth_toa_ranges(int device, int64_t n_filters, int n_anchors, const double *anchors_xyz,
                                      int n_epochs, const double *t, const kfpos_synth_toa *gen, int fmt,
                                      void *ranges, void *stream) {
    return synth_toa_ranges(device, n_filters, n_anchors, anchors_xyz, n_epochs, t, gen, fmt, ranges, nullptr, stream);
}

extern "C" int kfpos_synth_toa_ranges_nlos(int device, int64_t n_filters, int n_anchors, const double *anchors_xyz,
                                           int n_epochs, const double *t, const kfpos_synth_toa *gen, int fmt,
                                           void *ranges, uint32_t *nlos, void *stream) {
    if (!nlos) return KFPOS_ERR_INVALID;
    return synth_toa_ranges(device, n_filters, n_anchors, anchors_xyz, n_epochs, t, gen, fmt, ranges, nlos, stream);
}

namespace {
// how the selection of a T6 or ML batch is read from `sel` (used_mask): as the replay (T6) or the solve (ML, row 0
// of its [2][N]) wrote it
int sel_mode(const kfpos_batch *b) {
    const bool variant = b->cfg.variant == 1 || b->cfg.variant == 2;
    return variant ? SCORE_MASK : (b->model != KFPOS_MODEL_ML && b->cfg.ignore_worst_anchor) ? SCORE_LOO : SCORE_NONE;
}
} // namespace

extern "C" int kfpos_batch_score_selection(kfpos_batch *b, int n_rows, const void *ranges, int fmt, const int32_t *sel,
                                           const uint32_t *nlos, uint64_t *counts, void *stream) {
    static_assert(KFPOS_SCORE_COLS == SCORE_COLS, "one column count");
    if (!b) return KFPOS_ERR_INVALID;
    if (b->model == KFPOS_MODEL_K8 || b->model == KFPOS_MODEL_T9) return KFPOS_ERR_UNSUPPORTED;
    const bool ml = b->model == KFPOS_MODEL_ML;
    if (n_rows <= 0 || !fmt_ok(fmt) || !ranges || !counts || (ml && n_rows != 1)) return KFPOS_ERR_INVALID;
    if (!b->have_anchors) return KFPOS_ERR_NOT_READY;
    const int mode = sel_mode(b);
    if (mode != SCORE_NONE && !sel) return KFPOS_ERR_INVALID;
    DeviceGuard g(b->device);
    cudaStream_t s = (cudaStream_t)stream;
    const size_t N = (size_t)b->N, M = (size_t)b->anchors.n, R = (size_t)n_rows;
    Staging st(b, s);
    ScoreParams p;
    p.ranges = st.in(ranges, fmt_size(fmt) * M * N * R);
    p.sel = mode == SCORE_NONE ? nullptr : st.in(sel, sizeof(int32_t) * N * R);
    p.nlos = st.in(nlos, sizeof(uint32_t) * N * R);
    p.counts = (unsigned long long *)st.out(counts, sizeof(uint64_t) * SCORE_COLS * R);
    if (st.rc) return st.rc;
    p.N = b->N; p.n_rows = n_rows; p.M = (int)M; p.fmt = fmt; p.mode = mode;
    CK(cudaMemsetAsync(p.counts, 0, sizeof(uint64_t) * SCORE_COLS * R, s));
    CK(launch_score_selection(p, s));
    return st.finish();
}

extern "C" int kfpos_batch_crlb(kfpos_batch *b, int set, int n_rows, const double *truth, const void *ranges, int fmt,
                                double var_scalar, const double *var, const int32_t *sel, const uint32_t *nlos,
                                double *out, void *stream) {
    static_assert(KFPOS_CRLB_COLS == CRLB_W && KFPOS_CRLB_PRESENT == CRLB_PRESENT && KFPOS_CRLB_LOS == CRLB_LOS &&
                  KFPOS_CRLB_USED == CRLB_USED, "one set of constants");
    if (!b) return KFPOS_ERR_INVALID;
    const bool ml = b->model == KFPOS_MODEL_ML;
    if (set < KFPOS_CRLB_PRESENT || set > KFPOS_CRLB_USED || n_rows <= 0 || !fmt_ok(fmt) || !truth || !ranges ||
        !out || (!var && !(var_scalar > 0.0 && var_scalar < INFINITY)) || (set == KFPOS_CRLB_LOS && !nlos) ||
        (ml && n_rows != 1))
        return KFPOS_ERR_INVALID;
    if (set == KFPOS_CRLB_USED && (b->model == KFPOS_MODEL_K8 || b->model == KFPOS_MODEL_T9))
        return KFPOS_ERR_UNSUPPORTED;
    if (!b->have_anchors) return KFPOS_ERR_NOT_READY;
    const int mode = set == KFPOS_CRLB_USED ? sel_mode(b) : SCORE_NONE;
    if (mode != SCORE_NONE && !sel) return KFPOS_ERR_INVALID;
    DeviceGuard g(b->device);
    cudaStream_t s = (cudaStream_t)stream;
    const int64_t W = (b->N + 31) / 32;
    const size_t N = (size_t)b->N, M = (size_t)b->anchors.n, R = (size_t)n_rows;
    const size_t row_bytes = sizeof(double) * CRLB_W * (size_t)W;
    // the per-warp partials of a batch of rows, folded before the next batch: at most 256 MB of scratch
    int64_t batch_rows = (int64_t)(((size_t)256 << 20) / row_bytes);
    if (batch_rows < 1) batch_rows = 1;
    if (batch_rows > n_rows) batch_rows = n_rows;
    CK(b->crlb.reserve(row_bytes * (size_t)batch_rows));
    Staging st(b, s);
    CrlbParams p;
    p.anchors = b->anchors;
    const double *d_truth = st.in(truth, sizeof(double) * 3 * N * R);
    const char *d_ranges = (const char *)st.in(ranges, fmt_size(fmt) * M * N * R);
    const double *d_var = st.in(var, sizeof(double) * M * N * R);
    const int32_t *d_sel = mode == SCORE_NONE ? nullptr : st.in(sel, sizeof(int32_t) * N * R);
    const uint32_t *d_nlos = set == KFPOS_CRLB_LOS ? st.in(nlos, sizeof(uint32_t) * N * R) : nullptr;
    double *d_out = st.out(out, sizeof(double) * CRLB_W * R);
    if (st.rc) return st.rc;
    p.partials = (double *)b->crlb.p;
    p.w_scalar = var ? 0.0 : 1.0 / var_scalar;
    p.N = b->N; p.n_warps = W; p.M = (int)M; p.fmt = fmt; p.set = set; p.sel_mode = mode;
    p.dim = b->model == KFPOS_MODEL_K8 || (ml && b->cfg.use2d) ? 2 : 3;
    for (int64_t r0 = 0; r0 < n_rows; r0 += batch_rows) {
        const size_t o = (size_t)r0 * N;
        p.n_rows = n_rows - r0 < batch_rows ? n_rows - r0 : batch_rows;
        p.truth = d_truth + 3 * o;
        p.ranges = d_ranges + fmt_size(fmt) * M * o;
        p.var = d_var ? d_var + M * o : nullptr;
        p.sel = d_sel ? d_sel + o : nullptr;
        p.nlos = d_nlos ? d_nlos + o : nullptr;
        CK(launch_crlb(p, s));
        CK(launch_stats_tree(CRLB_W, p.n_rows, W, p.partials, p.partials, W * CRLB_W, CRLB_W, d_out + r0 * CRLB_W, s));
    }
    return st.finish();
}

extern "C" int kfpos_selftest_math(int device, int64_t n, const double *x, double *rcp, double *rsqrt, double *sn,
                                   double *cs) {
    if (n <= 0 || !x) return KFPOS_ERR_INVALID;
    if (int rc = check_device(device)) return rc;
    DeviceGuard g(device);
    if (!g.ok) return KFPOS_ERR_CUDA;
    Staging st(nullptr);
    st.sync = true; // a self-test returns the errors of its kernel, whatever the arrays
    const size_t bytes = 8 * (size_t)n;
    const double *d_x = st.in(x, bytes);
    double *d_rcp = st.out(rcp, bytes), *d_rsqrt = st.out(rsqrt, bytes), *d_sn = st.out(sn, bytes);
    double *d_cs = st.out(cs, bytes);
    if (st.rc) return st.rc;
    CK(launch_selftest_math(n, d_x, d_rcp, d_rsqrt, d_sn, d_cs, nullptr));
    return st.finish();
}

extern "C" int kfpos_selftest_ieee(int device, int64_t n, const double *a, const double *b, double *div_fast,
                                   double *div_ieee, double *sqrt_fast, double *sqrt_ieee, int32_t *flags) {
    if (n <= 0 || !a || !b) return KFPOS_ERR_INVALID;
    if (int rc = check_device(device)) return rc;
    DeviceGuard g(device);
    if (!g.ok) return KFPOS_ERR_CUDA;
    Staging st(nullptr);
    st.sync = true; // a self-test returns the errors of its kernel, whatever the arrays
    const size_t bytes = 8 * (size_t)n;
    const double *d_a = st.in(a, bytes), *d_b = st.in(b, bytes);
    double *d_df = st.out(div_fast, bytes), *d_di = st.out(div_ieee, bytes);
    double *d_sf = st.out(sqrt_fast, bytes), *d_si = st.out(sqrt_ieee, bytes);
    int32_t *d_flags = st.out(flags, 4 * (size_t)n);
    if (st.rc) return st.rc;
    CK(launch_selftest_ieee(n, d_a, d_b, d_df, d_di, d_sf, d_si, d_flags, nullptr));
    return st.finish();
}
