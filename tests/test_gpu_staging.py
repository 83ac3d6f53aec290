"""Host and device arguments of the C ABI.  Every entry point that takes data pointers gives bit-identical results
from numpy arrays, from CUDA tensors and from host inputs with device outputs; and the synchronisation rule of
include/kfpos_b200.h holds: a call given a host data array returns with its stream idle, a call given device data
arrays only (small HOST control arrays aside) returns with its work still queued."""
import ctypes as C

import numpy as np
import pytest

from roskfpos_b200 import lib as L, synth
from roskfpos_b200.batch import Batch
from tests.test_gpu_assemble import make_logs

pytestmark = pytest.mark.gpu

N, M, T = 37, 8, 5
MODES = ("host", "device", "host_in_device_out")
SLEEP_CYCLES = 100_000_000  # ~50 ms of torch.cuda._sleep ahead of the call under test


def ck(rc, what="call"):
    L.check(rc, what)


def hp(a):
    """Host pointer of a numpy array the caller keeps alive."""
    return C.c_void_p(a.ctypes.data)


class IO:
    """Where one run puts its arguments: numpy arrays on the host or torch tensors on cuda:0."""

    def __init__(self, mode):
        import torch
        self.torch = torch
        self.in_dev = mode == "device"
        self.out_dev = mode != "host"
        self.keep = []
        self.outs = {}

    def i(self, a, dev=None):
        a = np.ascontiguousarray(a)
        if self.in_dev if dev is None else dev:
            a = self.torch.as_tensor(a, device="cuda:0")
            self.keep.append(a)
            return C.c_void_p(a.data_ptr())
        self.keep.append(a)
        return hp(a)

    def o(self, name, shape, dtype=np.float64):
        assert name not in self.outs
        a = np.zeros(shape, dtype)
        if self.out_dev:
            a = self.torch.as_tensor(a, device="cuda:0")
            self.outs[name] = a
            return C.c_void_p(a.data_ptr())
        self.outs[name] = a
        return hp(a)

    def host_out(self, name, a):
        """A result that always lands in host memory (ctypes or numpy)."""
        self.outs[name] = np.frombuffer(bytes(a), dtype=np.uint8) if not isinstance(a, np.ndarray) else a

    def results(self):
        self.torch.cuda.synchronize()
        return {k: (v.cpu().numpy() if hasattr(v, "cpu") else v).copy() for k, v in self.outs.items()}


def _events(evs):
    arr = (L.KfposEvent * len(evs))()
    for i, ev in enumerate(evs):
        arr[i].kind, arr[i].dt, arr[i].offset = int(ev[0]), float(ev[1]), int(ev[2])
        for k, v in enumerate(ev[3] if len(ev) > 3 and ev[3] is not None else []):
            arr[i].aux[k] = float(v)
    return arr


def _t6_inputs():
    anc = synth.anchors_for(M)
    truth = synth.truth_lissajous(N, 3 * T + 1, 0.1)
    r = synth.ranges_mm(truth[1:], anc)
    x0 = np.vstack([truth[0], np.zeros((3, N))])
    P0 = np.zeros((6, 6, N))
    for k in range(6):
        P0[k, k] = 0.5 + 0.1 * k
    err = np.random.default_rng(1).uniform(0.005, 0.02, r.shape)
    dtf = np.full((T, N), 0.1)
    dtf[1, ::3] = -1.0
    return anc, truth, r, x0, P0.reshape(36, N), err, dtf


def run_t6(io):
    lib = L.lib()
    anc, truth, r, x0, P0, err, dtf = _t6_inputs()
    rows = 3 * T + 1
    dt = np.full(T, 0.1)
    with Batch(L.MODEL_T6, N, accel_noise=0.5, ignore_worst_anchor=1) as b:
        h = b._h
        ck(lib.kfpos_batch_set_anchors(h, M, io.i(anc)))
        ck(lib.kfpos_batch_set_state(h, io.i(x0), io.i(P0), None))
        ck(lib.kfpos_batch_set_truth_traj(h, rows, io.i(truth[1:]), None))
        # host ranges without per-ranging errors are streamed in chunks, with them they are staged whole
        ck(lib.kfpos_batch_replay_toa(h, T, hp(dt), io.i(r[:T]), L.FMT_I32_MM, 0.01, None, io.o("traj", (T, 3, N)),
                                      io.o("sel", (T, N), np.int32), None))
        ck(lib.kfpos_batch_replay_toa(h, T, hp(dt), io.i(r[T:2 * T]), L.FMT_I32_MM, 0.0, io.i(err[T:2 * T]),
                                      io.o("traj2", (T, 3, N)), io.o("sel2", (T, N), np.int32), None))
        ck(lib.kfpos_batch_replay_epochs(h, T, io.i(dtf), io.i(r[2 * T:3 * T]), L.FMT_I32_MM, 0.0,
                                         io.i(err[2 * T:3 * T]), io.o("traj3", (T, 3, N)), None))
        ck(lib.kfpos_batch_step_toa(h, 0.1, io.i(r[3 * T]), L.FMT_I32_MM, 0.01, None, None))
        ck(lib.kfpos_batch_get_state(h, io.o("x", (6, N)), io.o("P", (36, N)), io.o("status", N, np.int32), None))
        ck(lib.kfpos_batch_get_pose(h, 0.1, io.o("x_pred", (6, N)), io.o("P_pred", (36, N)), None))
        ck(lib.kfpos_batch_get_pose_msg(h, 0.1, io.o("pose", (13, N)), io.o("cov", (36, N)), None))
        ck(lib.kfpos_batch_epoch_stats(h, rows, io.o("epoch_stats", (rows, 6)), None))
        ck(lib.kfpos_batch_set_truth(h, io.i(truth[-1]), None))
        s1, s2, cnt = (C.c_double * 4)(), (C.c_double * 4)(), (C.c_double * 8)()
        ck(lib.kfpos_batch_error_stats(h, None, C.byref(s1), None))
        ck(lib.kfpos_batch_error_stats(h, io.i(truth[-2]), C.byref(s2), None))
        ck(lib.kfpos_batch_get_counters(h, C.byref(cnt), 0, None))
        io.host_out("error_stats_registered", s1)
        io.host_out("error_stats_given", s2)
        io.host_out("counters", cnt)
    return io.results()


def run_k8(io):
    lib = L.lib()
    anc = synth.anchors_for(M)
    w = synth.k8_workload(N, 2, anc, seed=synth.SEED + 3, full=True)
    evs = _events(w["events"])
    n_toa = sum(ev[0] == L.EV_TOA for ev in w["events"])
    rng = np.random.default_rng(2)
    dtf = np.array([[ev[1]] * N for ev in w["events"]])
    dtf[1, ::4] = -1.0
    srows = w["sensors"].shape[0]
    r = w["ranges"]
    with Batch(L.MODEL_K8, N, xml=synth.K8_XML, accel_noise=0.5, jolt=0.5) as b:
        h = b._h
        ck(lib.kfpos_batch_set_anchors(h, M, io.i(anc)))
        ck(lib.kfpos_batch_set_state(h, io.i(w["x0"]), None, None))
        ck(lib.kfpos_batch_replay_events(h, len(evs), C.cast(evs, C.c_void_p), io.i(r), L.FMT_I32_MM, 0.01, None,
                                         io.i(w["sensors"]), srows, io.o("traj", (n_toa, 3, N)), None))
        ck(lib.kfpos_batch_replay_events_ragged(h, len(evs), C.cast(evs, C.c_void_p), io.i(dtf), io.i(r),
                                                L.FMT_I32_MM, 0.01, None, io.i(w["sensors"]), srows,
                                                io.o("traj_ragged", (n_toa, 3, N)), None))
        px4 = [rng.normal(0.0, 0.01, N) for _ in range(3)] + [np.full(N, 33333.0)]
        ck(lib.kfpos_batch_step_px4(h, 0.033, *[io.i(a) for a in px4], io.i(np.full(N, 200, np.int32)), None))
        cov9 = np.diag([0.003, 0.003, 0.003]).reshape(9) + 0.0
        gyro9 = np.diag([0.089, 0.089, 0.089]).reshape(9) + 0.0
        ck(lib.kfpos_batch_step_imu(h, 0.01, io.i(rng.normal(0.0, 0.05, (3, N))), hp(gyro9),
                                    io.i(rng.normal(0.0, 0.1, (3, N))), hp(cov9), None))
        ang = rng.uniform(-3, 3, N)
        ck(lib.kfpos_batch_step_mag(h, 0.05, io.i(np.stack([np.cos(ang), np.sin(ang)])), None))
        ck(lib.kfpos_batch_step_compass(h, 0.05, io.i(ang), None))
        ck(lib.kfpos_batch_get_latches(h, io.o("latch", (16, N)), io.o("has", N, np.int32), io.o("latch_u", 16),
                                       None))
        latch, has, lu = np.ones((16, N)) * 0.25, np.full(N, 3, np.int32), np.full(16, 0.004)
        ck(lib.kfpos_batch_set_latches(h, io.i(latch), io.i(has), io.i(lu), None))
        # the K8 / T9 TOA-only schedules of replay_toa and replay_epochs
        ck(lib.kfpos_batch_replay_toa(h, 2, hp(np.full(2, 0.1)), io.i(r[:2]), L.FMT_I32_MM, 0.01, None,
                                      io.o("traj_toa", (2, 3, N)), None, None))
        ck(lib.kfpos_batch_replay_epochs(h, 2, io.i(dtf[:2]), io.i(r[:2]), L.FMT_I32_MM, 0.01, None,
                                         io.o("traj_epochs", (2, 3, N)), None))
        ck(lib.kfpos_batch_get_state(h, io.o("x", (8, N)), io.o("P", (64, N)), io.o("status", N, np.int32), None))
        ck(lib.kfpos_batch_get_pose_msg(h, 0.1, io.o("pose", (13, N)), io.o("cov", (36, N)), None))
    return io.results()


def run_t9(io):
    lib = L.lib()
    anc, truth, r, x0, _, _, _ = _t6_inputs()
    rng = np.random.default_rng(3)
    with Batch(L.MODEL_T9, N, accel_noise=0.5, jolt=0.5) as b:
        h = b._h
        ck(lib.kfpos_batch_set_anchors(h, M, io.i(anc)))
        ck(lib.kfpos_batch_set_state(h, io.i(np.vstack([x0, np.zeros((3, N))])), None, None))
        cov9 = np.diag([0.003, 0.003, 0.003]).reshape(9) + 0.0
        ck(lib.kfpos_batch_step_imu(h, 0.01, None, None, io.i(rng.normal(0.0, 0.1, (3, N))), hp(cov9), None))
        ck(lib.kfpos_batch_replay_toa(h, T, hp(np.full(T, 0.1)), io.i(r[:T]), L.FMT_I32_MM, 0.01, None,
                                      io.o("traj", (T, 3, N)), None, None))
        ck(lib.kfpos_batch_get_state(h, io.o("x", (9, N)), io.o("P", (81, N)), io.o("status", N, np.int32), None))
    return io.results()


def run_ml(io):
    lib = L.lib()
    anc, _, r, _, _, err, _ = _t6_inputs()
    with Batch(L.MODEL_ML, N, variant=2, use2d=0) as b:
        h = b._h
        ck(lib.kfpos_batch_set_anchors(h, M, io.i(anc)))
        ck(lib.kfpos_batch_ml_solve(h, io.i(r[0]), L.FMT_I32_MM, 0.0, io.i(err[0]), io.o("pos", (3, N)),
                                    io.o("cov", (9, N)), io.o("iters", N, np.int32), io.o("sel", (2, N), np.int32),
                                    io.o("status", N, np.int32), None))
    return io.results()


def run_no_handle(io):
    lib = L.lib()
    anc = synth.anchors_for(M)
    # epoch assembler
    anchor, seq, rmm, err, t = make_logs(N, 12, M, seed=4)
    Ta = 4 * 12 + 8
    ck(lib.kfpos_assemble_epochs_t(0, N, anchor.shape[0], M, io.i(anchor), io.i(seq), io.i(rmm), io.i(err), io.i(t),
                                   Ta, 0, 0.1, io.o("asm_ranges", (Ta, M, N), np.int32), io.o("asm_err", (Ta, M, N)),
                                   io.o("asm_dt", (Ta, N)), io.o("asm_n", N, np.int32), io.o("asm_t", (Ta, N)), None))
    # stream merger
    rng = np.random.default_rng(5)

    def arrivals(Lk, rate):
        tk = np.cumsum(rng.uniform(0.2, 1.8, (Lk, N)) * rate, axis=0).round(4)
        tk[np.arange(Lk)[:, None] >= rng.integers(0, Lk + 1, N)[None, :]] = -1.0
        return tk
    Tm = 6
    t_epoch, ranges = arrivals(Tm, 0.1), rng.integers(-1, 20000, (Tm, M, N)).astype(np.int32)
    errm = rng.uniform(0.01, 0.03, (Tm, M, N))
    sensors = {2: (arrivals(20, 0.03), rng.normal(size=(20, 3, N))), 1: (arrivals(8, 0.08), rng.normal(size=(8, 5, N))),
               4: (arrivals(5, 0.13), rng.normal(size=(5, 1, N)))}
    slots = np.array([2, 2, 1, 2, 0, 4, 3] * 5, dtype=np.int32)
    ns, tp, pp = (C.c_int64 * 4)(), (C.c_void_p * 4)(), (C.c_void_p * 4)()
    for k, (tk, pk) in sensors.items():
        ns[k - 1], tp[k - 1], pp[k - 1] = tk.shape[0], io.i(tk).value, io.i(pk).value
    n_rows = int((slots == L.EV_TOA).sum()) * M
    s_rows = int(sum(L.EV_ROWS[int(k)] for k in slots if k != L.EV_TOA))
    evs = (L.KfposEvent * len(slots))()
    aux = np.arange(9, dtype=np.float64)
    ck(lib.kfpos_merge_streams(0, N, M, Tm, io.i(t_epoch), io.i(ranges), io.i(errm), C.cast(ns, C.c_void_p),
                               C.cast(tp, C.c_void_p), C.cast(pp, C.c_void_p), len(slots), hp(slots), 0.1, hp(aux),
                               C.cast(evs, C.c_void_p), io.o("mrg_dt", (len(slots), N)),
                               io.o("mrg_ranges", (n_rows, N), np.int32), io.o("mrg_err", (n_rows, N)),
                               io.o("mrg_sensors", (s_rows, N)), io.o("mrg_dropped", N, np.int32), None))
    io.host_out("mrg_events", evs)
    # K8 generator: TOA, IMU, PX4, COMPASS, TOA
    kinds = [(L.EV_TOA, 0), (L.EV_IMU, 0), (L.EV_PX4, 3), (L.EV_COMPASS, 8), (L.EV_TOA, M)]
    sev = (L.KfposSynthEvent * len(kinds))()
    for i, (kind, off) in enumerate(kinds):
        sev[i].kind, sev[i].global_index, sev[i].t, sev[i].offset = kind, i, 0.02 * (i + 1), off
    ck(lib.kfpos_synth_k8(0, N, 3, C.c_uint64(7), M, io.i(anc), 1.049, 0.1, len(kinds), C.cast(sev, C.c_void_p),
                          0.12, 2 * M, 9, io.o("k8_ranges", (2 * M, N), np.int32), io.o("k8_sensors", (9, N)),
                          io.o("k8_x0", (8, N)), io.o("k8_truth_end", (3, N)), None))
    times = np.array([0.0, 0.05, 0.3])
    ck(lib.kfpos_synth_k8_truth(0, N, 3, C.c_uint64(7), len(times), io.i(times), 1.049,
                                io.o("k8_truth", (len(times), 3, N)), None))
    gen = L.KfposSynthToa(seed=9, first_filter=2, first_epoch=4, tag_z=1.0, sigma_r=0.1, p_missing=0.1, p_nlos=0.1,
                          nlos_mean=0.8)
    ck(lib.kfpos_synth_toa_ranges(0, N, M, io.i(anc), T, hp(np.arange(1, T + 1) * 0.1), C.byref(gen), L.FMT_I32_MM,
                                  io.o("toa_ranges", (T, M, N), np.int32), None))
    return io.results()


@pytest.mark.parametrize("scenario", [run_t6, run_k8, run_t9, run_ml, run_no_handle],
                         ids=lambda f: f.__name__[4:])
def test_host_and_device_arguments_agree(kflib, scenario):
    got = {mode: scenario(IO(mode)) for mode in MODES}
    ref = got["host"]
    for mode in MODES[1:]:
        assert got[mode].keys() == ref.keys()
        for k in ref:
            assert got[mode][k].dtype == ref[k].dtype and got[mode][k].tobytes() == ref[k].tobytes(), (mode, k)


def _busy_after(call, stream, warm=1):
    """Runs `call` behind a ~50 ms sleep on `stream`; True if the stream still has work when the call returns.
    `warm` calls come first: growing a scratch slot frees the old one, and cudaFree synchronises the device."""
    import torch
    for _ in range(warm):
        call()
    stream.synchronize()
    with torch.cuda.stream(stream):
        torch.cuda._sleep(SLEEP_CYCLES)
    call()
    busy = not stream.query()
    stream.synchronize()
    return busy


def test_host_data_arrays_synchronise(kflib):
    import torch
    lib = L.lib()
    s = torch.cuda.Stream()
    sp = C.c_void_p(s.cuda_stream)
    dev = lambda a: torch.as_tensor(np.ascontiguousarray(a), device="cuda:0")
    dp = lambda t: C.c_void_p(t.data_ptr())
    anc, truth, r, x0, _, err, _ = _t6_inputs()
    w = synth.k8_workload(N, 1, anc, seed=synth.SEED + 3, full=True)
    evs = _events(w["events"])
    dtf = np.array([[ev[1]] * N for ev in w["events"]])
    srows = w["sensors"].shape[0]
    rows = [np.full(N, 0.01) for _ in range(4)]
    q = np.full(N, 200, np.int32)
    acc, gyro, mag, cmp = np.full((3, N), 0.01), np.full((3, N), 0.02), np.ones((2, N)), np.zeros(N)
    with Batch(L.MODEL_K8, N, anchors=anc, xml=synth.K8_XML, accel_noise=0.5, jolt=0.5) as b:
        b.set_state(w["x0"])
        h = b._h
        calls = {
            "step_px4": lambda: lib.kfpos_batch_step_px4(h, 0.033, *[hp(a) for a in rows], hp(q), sp),
            "step_imu": lambda: lib.kfpos_batch_step_imu(h, 0.01, hp(gyro), None, hp(acc), None, sp),
            "step_mag": lambda: lib.kfpos_batch_step_mag(h, 0.05, hp(mag), sp),
            "step_compass": lambda: lib.kfpos_batch_step_compass(h, 0.05, hp(cmp), sp),
            "replay_events": lambda: lib.kfpos_batch_replay_events(
                h, len(evs), C.cast(evs, C.c_void_p), hp(w["ranges"]), L.FMT_I32_MM, 0.01, None, hp(w["sensors"]),
                srows, None, sp),
            "replay_events_ragged": lambda: lib.kfpos_batch_replay_events_ragged(
                h, len(evs), C.cast(evs, C.c_void_p), hp(dtf), hp(w["ranges"]), L.FMT_I32_MM, 0.01, None,
                hp(w["sensors"]), srows, None, sp),
        }
        for name, call in calls.items():
            assert not _busy_after(lambda: ck(call(), name), s), name
    d_r, d_out = dev(r[0]), [torch.zeros((k, N), dtype=dt, device="cuda:0")
                             for k, dt in ((3, torch.float64), (9, torch.float64), (1, torch.int32),
                                           (2, torch.int32), (1, torch.int32))]
    e0 = np.ascontiguousarray(err[0])
    with Batch(L.MODEL_ML, N, anchors=anc) as b:  # only err_var on the host
        assert not _busy_after(lambda: ck(lib.kfpos_batch_ml_solve(b._h, dp(d_r), L.FMT_I32_MM, 0.0, hp(e0),
                                                                   *[dp(o) for o in d_out], sp)), s)
    tr = np.ascontiguousarray(truth[-1])
    with Batch(L.MODEL_T6, N, anchors=anc, accel_noise=0.5) as b:  # a host truth, the result stays on the device
        b.set_state(x0)
        assert not _busy_after(lambda: ck(lib.kfpos_batch_error_stats(b._h, hp(tr), None, sp)), s)
    torch.cuda.synchronize()


def test_device_data_arrays_stay_asynchronous(kflib):
    import torch
    lib = L.lib()
    s = torch.cuda.Stream()
    sp = C.c_void_p(s.cuda_stream)
    dev = lambda a: torch.as_tensor(np.ascontiguousarray(a), device="cuda:0")
    dp = lambda t: C.c_void_p(t.data_ptr())
    anc, truth, r, x0, P0, _, _ = _t6_inputs()
    d_r, d_x0, d_P0, d_truth = dev(r[:T]), dev(x0), dev(P0.reshape(6, 6, N)), dev(truth[-1])
    dt = np.full(T, 0.1)  # a HOST control array: it does not make the call synchronise
    with Batch(L.MODEL_T6, N, anchors=anc, accel_noise=0.5) as b:
        h = b._h
        assert _busy_after(lambda: ck(lib.kfpos_batch_set_state(h, dp(d_x0), dp(d_P0), sp)), s)
        assert _busy_after(lambda: ck(lib.kfpos_batch_replay_toa(h, T, hp(dt), dp(d_r), L.FMT_I32_MM, 0.01, None,
                                                                 None, None, sp)), s)
        ck(lib.kfpos_batch_set_truth(h, dp(d_truth), sp))
        assert _busy_after(lambda: ck(lib.kfpos_batch_error_stats(h, None, None, sp)), s)
    gen = L.KfposSynthToa(seed=9, first_filter=0, first_epoch=0, tag_z=1.0, sigma_r=0.1)
    t = np.arange(1, T + 1) * 0.1
    d_ranges = torch.empty((T, M, N), dtype=torch.int32, device="cuda:0")
    assert _busy_after(lambda: ck(lib.kfpos_synth_toa_ranges(0, N, M, hp(anc), T, hp(t), C.byref(gen), L.FMT_I32_MM,
                                                             dp(d_ranges), sp)), s)
    sev = (L.KfposSynthEvent * 2)()
    for i in range(2):
        sev[i].kind, sev[i].global_index, sev[i].t, sev[i].offset = L.EV_TOA, i, 0.1 * (i + 1), i * M
    d_k8 = torch.empty((2 * M, N), dtype=torch.int32, device="cuda:0")
    d_end = torch.empty((3, N), dtype=torch.float64, device="cuda:0")
    # warm every slot of the generator's 8-slot event ring: growing one synchronises the device
    assert _busy_after(lambda: ck(lib.kfpos_synth_k8(0, N, 0, C.c_uint64(1), M, hp(anc), 1.049, 0.1, 2,
                                                     C.cast(sev, C.c_void_p), 0.2, 2 * M, 0, dp(d_k8), None, None,
                                                     dp(d_end), sp)), s, warm=8)
    torch.cuda.synchronize()
