"""Synthetic workloads for the BASELINE.json configs (SURVEY.md §8d).

Host-side (numpy) generators used by the parity tests -- the same arrays are fed
to the CPU oracle and to the CUDA library -- and device-side (torch) generators
used by bench.py to fill HBM with inputs of the full BASELINE sizes.  Ranges are
produced in the reference's own wire format: integer millimetres, floored
(PG.cpp:213), with <= 0 meaning "no ranging from this anchor" (PG.cpp:482,
TOA.cpp:50).
"""
from __future__ import annotations

import numpy as np

SEED = 20190816  # base seed, SURVEY.md §8d


def anchors_for(n_anchors: int) -> np.ndarray:
    """Anchor tables of the BASELINE configs, [n][3] float64 metres."""
    if n_anchors == 4:  # config 1: non-coplanar so the 3-D ML is well posed
        a = [(0, 0, 2.5), (10, 0, 0.5), (10, 10, 2.5), (0, 10, 0.5)]
    elif n_anchors == 8:  # config 2/3/5: perimeter of a 10 x 10 m room, z alternating
        xy = [(0, 0), (5, 0), (10, 0), (10, 5), (10, 10), (5, 10), (0, 10), (0, 5)]
        a = [(x, y, 0.5 if i % 2 else 2.5) for i, (x, y) in enumerate(xy)]
    elif n_anchors == 16:  # config 4: 4 x 4 grid, ceiling/floor alternating
        a = []
        for i in range(4):
            for j in range(4):
                a.append((10.0 * i / 3, 10.0 * j / 3, 2.5 if (i + j) % 2 == 0 else 0.5))
    else:
        rng = np.random.default_rng(SEED + n_anchors)
        a = np.column_stack([rng.uniform(0, 10, n_anchors), rng.uniform(0, 10, n_anchors),
                             rng.uniform(0.3, 2.7, n_anchors)])
    return np.ascontiguousarray(np.asarray(a, dtype=np.float64))


def truth_lissajous(n_filters: int, n_steps: int, dt: float, seed: int = SEED, z: float = 1.0):
    """Per-filter Lissajous truth, returns pos [T+1][3][N] (index 0 = initial position)."""
    rng = np.random.default_rng(seed)
    ph = rng.uniform(0, 2 * np.pi, size=(2, n_filters))
    t = (np.arange(n_steps + 1) * dt)[:, None]
    x = 5 + 3 * np.sin(0.20 * t + ph[0][None, :])
    y = 5 + 3 * np.sin(0.31 * t + ph[1][None, :])
    zz = np.full_like(x, z)
    return np.ascontiguousarray(np.stack([x, y, zz], axis=1))


def ranges_mm(truth: np.ndarray, anchors: np.ndarray, sigma: float = 0.10, seed: int = SEED + 1,
              p_missing: float = 0.0, p_nlos: float = 0.0, nlos_mean: float = 0.8,
              dtype=np.int32) -> np.ndarray:
    """Noisy floored-mm ranges [T][M][N] for truth [T][3][N] (or [3][N] -> [M][N])."""
    rng = np.random.default_rng(seed)
    single = truth.ndim == 2
    tr = truth[None] if single else truth
    d = np.sqrt(((tr[:, None, :, :] - anchors[None, :, :, None]) ** 2).sum(axis=2))  # [T][M][N]
    r = d + rng.normal(0.0, sigma, size=d.shape)
    if p_nlos > 0:
        nl = rng.random(size=d.shape) < p_nlos
        r = r + nl * rng.exponential(nlos_mean, size=d.shape)
    mm = np.floor(r * 1000.0)
    if p_missing > 0:
        mm[rng.random(size=d.shape) < p_missing] = 0
    mm = np.clip(mm, 0, np.iinfo(dtype).max).astype(dtype)
    return np.ascontiguousarray(mm[0] if single else mm)


EV_TOA, EV_PX4, EV_IMU, EV_MAG, EV_COMPASS = 0, 1, 2, 3, 4
# per 0.1 s macro-step (BASELINE configs 3 and 5, SURVEY.md §8d): 10 IMU samples, 1 compass,
# 1 TOA epoch (+ 3 PX4Flow frames for the full multi-sensor config); dt sums to 0.1 s and is
# never 0 (px4flowOutput divides by timeLag, KF.cpp:566)
MACRO_IMU_MAG = [(EV_IMU, 0.009)] * 10 + [(EV_COMPASS, 0.005), (EV_TOA, 0.005)]
MACRO_FULL = ([(EV_IMU, 0.008)] * 3 + [(EV_PX4, 0.003)] + [(EV_IMU, 0.008)] * 3 + [(EV_PX4, 0.003)] +
              [(EV_IMU, 0.008)] * 4 + [(EV_PX4, 0.003)] + [(EV_COMPASS, 0.005), (EV_TOA, 0.006)])
IMU_AUX = [0.003, 0.0, 0.0, 0.003, 0.089]  # cov_acc[0],[1],[3],[4], cov_ang_vel[8] (config_imu.xml:2)
PX4_HEIGHT, PX4_T_US = 5.0, 33333.0      # config_px4flow.xml:2


def k8_workload(n_filters, n_macro, anchors, seed=SEED, full=False, sigma_r=0.10, xp=None, device=None):
    """Multi-sensor event stream for KalmanFilter (K8) batches.

    Returns dict(events=[(kind, dt, offset_row, aux)], ranges int32 [T][M][N], sensors f64 [R][N],
    x0 [8][N], truth_end [3][N] (x, y, tag z)).  `xp` = numpy (default) or torch (then `device`).
    """
    macro = MACRO_FULL if full else MACRO_IMU_MAG
    use_torch = xp is not None and xp.__name__ == "torch"
    if use_torch:
        import torch
        g = torch.Generator(device=device)
        g.manual_seed(seed)
        f64 = dict(device=device, dtype=torch.float64)
        rand = lambda *s: torch.rand(*s, generator=g, **f64)
        randn = lambda *s: torch.randn(*s, generator=g, **f64)
        sin, cos, sqrt, floor, stack = torch.sin, torch.cos, torch.sqrt, torch.floor, torch.stack
        anc = torch.as_tensor(anchors, **f64)
        full_like = lambda a, v: torch.full_like(a, v)
    else:
        rng = np.random.default_rng(seed)
        rand = lambda *s: rng.random(s)
        randn = lambda *s: rng.normal(size=s)
        sin, cos, sqrt, floor, stack = np.sin, np.cos, np.sqrt, np.floor, np.stack
        anc = np.asarray(anchors, dtype=np.float64)
        full_like = lambda a, v: np.full_like(a, v)
    N, M = n_filters, len(anchors)
    ph = rand(2, N) * (2 * np.pi)
    th0 = 0.3 + 0.2 * rand(N)
    om = 0.05
    tag_z = 1.049

    def kin(t):
        px = 5 + 3 * sin(0.20 * t + ph[0]); py = 5 + 3 * sin(0.31 * t + ph[1])
        vx = 0.6 * cos(0.20 * t + ph[0]); vy = 0.93 * cos(0.31 * t + ph[1])
        ax = -0.12 * sin(0.20 * t + ph[0]); ay = -0.2883 * sin(0.31 * t + ph[1])
        return px, py, vx, vy, ax, ay, th0 + om * t

    events, rows, rng_rows = [], [], []
    t = 0.0
    for _ in range(n_macro):
        for kind, dt in macro:
            t += dt
            px, py, vx, vy, ax, ay, th = kin(t)
            c, s = cos(th), sin(th)
            if kind == EV_TOA:
                d = sqrt((px[None] - anc[:, 0:1]) ** 2 + (py[None] - anc[:, 1:2]) ** 2 + (tag_z - anc[:, 2:3]) ** 2)
                d = d + sigma_r * randn(M, N)
                events.append((kind, dt, len(rng_rows) * M, None))
                rng_rows.append(floor(d * 1000.0))
            elif kind == EV_IMU:
                off = len(rows)
                rows.append(om + np.sqrt(0.089) * randn(N))
                rows.append(c * ax + s * ay + np.sqrt(0.003) * randn(N))
                rows.append(-s * ax + c * ay + np.sqrt(0.003) * randn(N))
                events.append((kind, dt, off, IMU_AUX))
            elif kind == EV_PX4:
                off = len(rows)
                T = PX4_T_US / 1e6
                rows.append((c * vx + s * vy) * T / PX4_HEIGHT + 2e-4 * randn(N))
                rows.append((-s * vx + c * vy) * T / PX4_HEIGHT + 2e-4 * randn(N))
                rows.append(full_like(px, om * T))
                rows.append(full_like(px, PX4_T_US))
                rows.append(full_like(px, 200.0))
                events.append((kind, dt, off, None))
            else:
                off = len(rows)
                a = th + 0.01 * randn(N)
                rows.append(a - 2 * np.pi * floor((a + np.pi) / (2 * np.pi)))
                events.append((kind, dt, off, None))
    px, py, vx, vy, ax, ay, th = kin(0.0)
    zeros = full_like(px, 0.0)
    x0 = stack([px, py, vx, vy, zeros, zeros, th, full_like(px, om)])
    pe = kin(t)
    truth_end = stack([pe[0], pe[1], full_like(px, tag_z)])
    ranges = stack(rng_rows)
    sensors = stack(rows)
    if use_torch:
        import torch
        ranges = ranges.clamp_(min=0).to(torch.int32).contiguous()
        sensors = sensors.contiguous()
    else:
        ranges = np.ascontiguousarray(np.clip(ranges, 0, None).astype(np.int32))
        sensors = np.ascontiguousarray(sensors)
    return dict(events=events, ranges=ranges, sensors=sensors, x0=x0, truth_end=truth_end, tag_z=tag_z,
                n_toa=len(rng_rows), n_events=len(events))


K8_XML = ['<config><uwb useFixedHeight="0" fixedHeight="1.049" tagId="0"/></config>',
          '<config><px4flow armP0="1" armP1="0" useFixedSensorHeight="1" sensorHeight="5" '
          'sensorInitAngle="-1.570796326794897" covarianceVelocity="0.04" covarianceGyroZ="0.02"/></config>',
          '<config><imu useFixedCovarianceAcceleration="1" covarianceAcceleration="0.003" '
          'useFixedCovarianceAngularVelocityZ="1" covarianceAngularVelocityZ="0.089"/></config>',
          '<config><mag angleOffset="0" covarianceMag="0.0001"/></config>']
K8_ORACLE_CFG = dict(tag_z=1.049, use_fixed_height=0, px4_height=5.0, px4_arm1=1.0, px4_arm2=0.0,
                     px4_cov_vel=0.04, px4_cov_gyro=0.02, imu_fixed_cov_acc=1, imu_cov_acc=0.003,
                     imu_fixed_cov_gyro=1, imu_cov_gyro=0.089, mag_offset=0.0, mag_cov=1e-4)


def device_ranges_mm(n_filters: int, n_steps: int, anchors: np.ndarray, dt: float, device,
                     seed: int = SEED, sigma: float = 0.10, dtype=None, step0: int = 0):
    """torch/device version of truth_lissajous + ranges_mm for bench-sized inputs.

    Returns (ranges [T][M][N] int32 on `device`, x0 [3][N] float64, truth_end [3][N]).
    The inputs are i.i.d. per filter; only their shape/statistics matter to the bench.
    """
    import torch

    g = torch.Generator(device=device)
    g.manual_seed(seed)
    dtype = dtype or torch.int32
    ph = torch.rand((2, n_filters), generator=g, device=device, dtype=torch.float64) * (2 * np.pi)
    anc = torch.as_tensor(anchors, device=device, dtype=torch.float64)
    m = anc.shape[0]
    out = torch.empty((n_steps, m, n_filters), device=device, dtype=dtype)

    def pos(k):
        t = k * dt
        return torch.stack([5 + 3 * torch.sin(0.20 * t + ph[0]), 5 + 3 * torch.sin(0.31 * t + ph[1]),
                            torch.ones_like(ph[0])])

    x0 = pos(step0)
    p = x0
    for k in range(n_steps):
        p = pos(step0 + k + 1)
        d = torch.sqrt(((p[None, :, :] - anc[:, :, None]) ** 2).sum(dim=1))  # [M][N]
        d = d + sigma * torch.randn(d.shape, generator=g, device=device, dtype=torch.float64)
        out[k] = torch.floor(d * 1000.0).clamp_(min=0).to(dtype)
    return out, x0.contiguous(), p.contiguous()


def device_truth_traj(n_filters: int, n_steps: int, dt: float, device, seed: int = SEED, step0: int = 0):
    """The per-step truth of device_ranges_mm with the same arguments (same generator, same first draw, so the
    same phases): SoA [T][3][N] float64 on `device`, row k = the position at step step0 + k + 1 -- the truth
    of the replay's output row k, for Batch.set_truth_traj."""
    import torch

    g = torch.Generator(device=device)
    g.manual_seed(seed)
    ph = torch.rand((2, n_filters), generator=g, device=device, dtype=torch.float64) * (2 * np.pi)
    out = torch.empty((n_steps, 3, n_filters), device=device, dtype=torch.float64)
    for k in range(n_steps):
        t = (step0 + k + 1) * dt
        out[k, 0] = 5 + 3 * torch.sin(0.20 * t + ph[0])
        out[k, 1] = 5 + 3 * torch.sin(0.31 * t + ph[1])
        out[k, 2] = 1.0
    return out


def k8_montecarlo_chunk(n_filters, macro0, n_macro, anchors, device, seed=SEED, full=False, sigma_r=0.10,
                        first_filter=0, want_x0=False, out=None, stream=None, want_truth_toa=False):
    """Macro-steps [macro0, macro0 + n_macro) of the K8 Monte Carlo workload, generated ON THE DEVICE by
    kfpos_synth_k8 (Philox4x32-10; the stream of a filter depends only on seed, its global index and the
    global event index).  Returns the dict k8_workload returns (events for replay_events, ranges int32
    [T][M][N], sensors f64 [R][N], truth_end [3][N], x0 [8][N] if want_x0) with torch tensors on `device`;
    `out` may hold the tensors of a previous chunk of the same shape to be reused.  want_truth_toa: also
    truth_toa [n_toa][3][N], the truth (x, y, tag z) at the chunk's TOA events made on the device by
    kfpos_synth_k8_truth -- what Batch.set_truth_traj takes for the per-epoch statistics of the chunk."""
    import ctypes as C
    import torch
    from . import lib as L
    from .batch import _stream_ptr
    macro = MACRO_FULL if full else MACRO_IMU_MAG
    M, N = len(anchors), int(n_filters)
    rows_of = {EV_IMU: 3, EV_PX4: 5, EV_COMPASS: 1}
    # event times from integer milliseconds, so that they do not depend on where a chunk starts
    cum_ms = np.cumsum([int(round(dt * 1000)) for _, dt in macro])
    macro_ms = int(cum_ms[-1])
    t = 0.0
    events, sev = [], []
    n_rng = n_sens = 0
    for mstep in range(n_macro):
        for j, (kind, dt) in enumerate(macro):
            t = ((macro0 + mstep) * macro_ms + int(cum_ms[j])) / 1000.0
            g = (macro0 + mstep) * len(macro) + j
            if kind == EV_TOA:
                off = n_rng * M; n_rng += 1
                events.append((kind, dt, off, None))
            else:
                off = n_sens; n_sens += rows_of[kind]
                events.append((kind, dt, off, IMU_AUX if kind == EV_IMU else None))
            sev.append((kind, g, t, off))
    dev = torch.device(device)
    if out is None:
        out = {}
    def buf(name, shape, dtype):
        tns = out.get(name)
        if tns is None or tuple(tns.shape) != tuple(shape):
            tns = torch.empty(shape, device=dev, dtype=dtype)
        return tns
    ranges = buf("ranges", (n_rng, M, N), torch.int32)
    sensors = buf("sensors", (n_sens, N), torch.float64)
    truth_end = buf("truth_end", (3, N), torch.float64)
    x0 = buf("x0", (8, N), torch.float64) if want_x0 else None
    arr = (L.KfposSynthEvent * len(sev))()
    for i, (kind, g, tt, off) in enumerate(sev):
        arr[i].kind, arr[i].global_index, arr[i].t, arr[i].offset = int(kind), int(g), float(tt), int(off)
    anc = np.ascontiguousarray(anchors, dtype=np.float64)
    sp = _stream_ptr(stream)
    L.check(L.lib().kfpos_synth_k8(dev.index or 0, N, int(first_filter), C.c_uint64(seed), M,
                                   C.c_void_p(anc.ctypes.data), 1.049, float(sigma_r), len(sev),
                                   C.cast(arr, C.c_void_p), float(t), n_rng * M, n_sens,
                                   C.c_void_p(ranges.data_ptr()), C.c_void_p(sensors.data_ptr()),
                                   None if x0 is None else C.c_void_p(x0.data_ptr()),
                                   C.c_void_p(truth_end.data_ptr()), sp), "kfpos_synth_k8")
    res = dict(events=events, ranges=ranges, sensors=sensors, x0=x0, truth_end=truth_end, tag_z=1.049,
               n_toa=n_rng, n_events=len(events))
    if want_truth_toa:
        t_toa = np.ascontiguousarray([tt for kind, _, tt, _ in sev if kind == EV_TOA], dtype=np.float64)
        truth_toa = buf("truth_toa", (n_rng, 3, N), torch.float64)
        L.check(L.lib().kfpos_synth_k8_truth(dev.index or 0, N, int(first_filter), C.c_uint64(seed), n_rng,
                                             C.c_void_p(t_toa.ctypes.data), 1.049, C.c_void_p(truth_toa.data_ptr()), sp),
                "kfpos_synth_k8_truth")
        res["truth_toa"] = truth_toa
    return res


def walk_truth_chunk(n_filters, epoch0, n_epochs, device, *, seed, period, accel_sd, v_max, lo, hi, first_filter=0,
                     state=None, want_x0=False, out=None, stream=None):
    """Epochs [epoch0, epoch0 + n_epochs) of the random walk of kfpos_synth_walk (DESIGN §4.5g), generated ON THE
    DEVICE: discrete white-noise acceleration of sd accel_sd (m/s^2, per axis) with speeds capped at v_max (m/s, per
    axis, inf: no cap), reflected at the walls of the box [lo, hi] (m).  An axis with accel_sd 0 stays at the
    centre of the box (a fixed tag height).  Each position is a pure function of (seed, first_filter + f, epoch)
    and the state the chunk starts from, so sharding and chunking change nothing.
    state: None draws the initial state (zero velocity, uniform in the box); else the [6][N] float64 device tensor
    (x, y, z, vx, vy, vz, the T6 state layout) at epoch0, which the call advances IN PLACE to the state after the
    last epoch.  Returns dict(truth [n_epochs][3][N] float64 on `device`, row k the position at time
    (epoch0 + k + 1) * period, what toa_montecarlo_chunk(truth=...) and Batch.set_truth_traj take; state [6][N];
    x0 [6][N] the initial state when state is None and want_x0).  `out` may hold the tensors of a previous chunk of
    the same shape to be reused."""
    import ctypes as C
    import torch
    from . import lib as L
    from .batch import _stream_ptr
    N, n = int(n_filters), int(n_epochs)
    dev = torch.device(device)
    out = {} if out is None else out

    def buf(name, shape):
        tns = out.get(name)
        if tns is None or tuple(tns.shape) != tuple(shape) or tns.dtype != torch.float64:
            tns = out[name] = torch.empty(shape, device=dev, dtype=torch.float64)
        return tns
    vec = lambda v: np.broadcast_to(np.asarray(v, dtype=np.float64), (3,))
    w = L.KfposSynthWalk(seed=int(seed), first_filter=int(first_filter), first_epoch=int(epoch0), period=float(period))
    w.accel_sd[:], w.v_max[:], w.lo[:], w.hi[:] = vec(accel_sd), vec(v_max), vec(lo), vec(hi)
    truth = buf("truth", (n, 3, N))
    sp = _stream_ptr(stream)

    def call(init, n_ep, st):
        w.init = init
        L.check(L.lib().kfpos_synth_walk(dev.index or 0, N, n_ep, C.byref(w), C.c_void_p(st.data_ptr()),
                                         C.c_void_p(truth.data_ptr()) if n_ep else None, sp), "kfpos_synth_walk")
    res = dict(truth=truth)
    if state is None:
        state = buf("state", (6, N))
        if want_x0:  # the initial state on its own, then the epochs from it: the same numbers as one init call
            x0 = buf("x0", (6, N))
            call(1, 0, x0)
            state.copy_(x0)
            res["x0"] = x0
            call(0, n, state)
        else:
            call(1, n, state)
    else:
        if tuple(state.shape) != (6, N) or state.dtype != torch.float64 or not state.is_cuda:
            raise ValueError("walk_truth_chunk: state must be a [6][N] float64 device tensor")
        call(0, n, state)
    res["state"] = state
    return res


def toa_montecarlo_chunk(n_filters, epoch0, n_epochs, anchors, device, seed=SEED, period=0.1, sigma_r=0.10,
                         p_missing=0.0, p_nlos=0.0, nlos_mean=0.8, tag_z=1.0, first_filter=0, fmt=None,
                         want_x0=False, want_truth=False, out=None, stream=None, want_nlos=False, obstacles=None,
                         truth=None):
    """Ranging epochs [epoch0, epoch0 + n_epochs) of the T6 Monte Carlo workload, generated ON THE DEVICE by
    kfpos_synth_toa_ranges (Philox4x32-10; a ranging depends only on seed, the global filter index
    first_filter + f, the global epoch index and the anchor, so sharding and chunking change nothing).  Epoch k
    is at t[k] = (epoch0 + k + 1) * period; the truth is the Lissajous of kfpos_synth_k8 at height tag_z.
    p_missing: probability that a ranging is absent (written as 0); p_nlos: probability of a positive NLOS
    bias, exponential with mean nlos_mean (m).  fmt: lib.FMT_I32_MM (default) or lib.FMT_U16_MM.

    Returns dict(ranges [n][M][N] on `device`, dt = period, t (host [n]), truth_end [3][N] = the truth at
    t[-1], x0 [6][N] (the truth at t = 0 with zero velocity, a T6 state) if want_x0, truth [n][3][N] (from
    kfpos_synth_k8_truth, what Batch.set_truth_traj takes for the chunk) if want_truth, nlos [n][N] if want_nlos:
    the NLOS ground truth of kfpos_synth_toa_ranges_nlos, bit a set where ranging a carries a bias and is present,
    as int32 holding the uint32 bits).  `out` may hold the tensors of a previous chunk of the same shape to be
    reused.  ML batches take `ranges` row by row.
    obstacles: [n][9] boxes (lo x y z, hi x y z, excess_per_m, spread, p_loss; DESIGN §4.5f) whose crossing biases
    or removes a ranging (kfpos_synth_toa_ranges_geo); the nlos mask then also marks the blocked rangings.  None or
    an empty array: no boxes, the calls above.
    truth: a [n_epochs][3][N] float64 device tensor of positions (walk_truth_chunk, or any trajectory; DESIGN §4.5g)
    in place of the Lissajous: the rangings come from kfpos_synth_toa_ranges_truth (tag_z is ignored), boxes and
    the mask work as above, want_truth returns this tensor and truth_end is its last row.  want_x0 then has no
    Lissajous to start from and is refused (walk_truth_chunk gives a walk's x0)."""
    import ctypes as C
    import torch
    from . import lib as L
    from .batch import _stream_ptr
    fmt = L.FMT_I32_MM if fmt is None else int(fmt)
    if fmt not in (L.FMT_I32_MM, L.FMT_U16_MM):
        raise ValueError("toa_montecarlo_chunk: fmt must be FMT_I32_MM or FMT_U16_MM")
    anc = np.ascontiguousarray(anchors, dtype=np.float64).reshape(-1, 3)
    M, N, n = len(anc), int(n_filters), int(n_epochs)
    if truth is not None:
        if tuple(truth.shape) != (n, 3, N) or truth.dtype != torch.float64 or not truth.is_cuda:
            raise ValueError("toa_montecarlo_chunk: truth must be a [n_epochs][3][N] float64 device tensor")
        if want_x0:
            raise ValueError("toa_montecarlo_chunk: want_x0 needs the Lissajous; walk_truth_chunk gives a walk's x0")
        truth = truth.contiguous()
    # times from the global epoch index, so that they do not depend on where a chunk starts
    t = np.ascontiguousarray(np.arange(epoch0 + 1, epoch0 + n + 1, dtype=np.float64) * period)
    dev = torch.device(device)
    out = {} if out is None else out

    def buf(name, shape, dtype):
        tns = out.get(name)
        if tns is None or tuple(tns.shape) != tuple(shape) or tns.dtype != dtype:
            tns = out[name] = torch.empty(shape, device=dev, dtype=dtype)
        return tns
    ranges = buf("ranges", (n, M, N), torch.uint16 if fmt == L.FMT_U16_MM else torch.int32)
    gen = L.KfposSynthToa(seed=int(seed), first_filter=int(first_filter), first_epoch=int(epoch0), tag_z=float(tag_z),
                          sigma_r=float(sigma_r), p_missing=float(p_missing), p_nlos=float(p_nlos),
                          nlos_mean=float(nlos_mean))
    sp = _stream_ptr(stream)
    args = (dev.index or 0, N, M, C.c_void_p(anc.ctypes.data), n, C.c_void_p(t.ctypes.data), C.byref(gen), fmt,
            C.c_void_p(ranges.data_ptr()))
    nlos = buf("nlos", (n, N), torch.int32) if want_nlos else None  # torch has no general uint32: the mask bits
    box = np.zeros((0, 9)) if obstacles is None else np.asarray(obstacles, dtype=np.float64).reshape(-1, 9)
    tbl = None
    if len(box):
        tbl = (L.KfposObstacle * len(box))()
        for o, b in zip(tbl, box):
            o.lo[:], o.hi[:] = b[0:3], b[3:6]
            o.excess_per_m, o.spread, o.p_loss = b[6], b[7], b[8]
        tbl = C.cast(tbl, C.c_void_p)
    if truth is not None:
        targs = args[:5] + (C.c_void_p(truth.data_ptr()),) + args[6:]
        L.check(L.lib().kfpos_synth_toa_ranges_truth(*targs[:7], len(box), tbl, *targs[7:],
                                                     None if nlos is None else C.c_void_p(nlos.data_ptr()), sp),
                "kfpos_synth_toa_ranges_truth")
    elif len(box):
        L.check(L.lib().kfpos_synth_toa_ranges_geo(*args[:7], len(box), tbl, *args[7:],
                                                   None if nlos is None else C.c_void_p(nlos.data_ptr()), sp),
                "kfpos_synth_toa_ranges_geo")
    elif want_nlos:
        L.check(L.lib().kfpos_synth_toa_ranges_nlos(*args, C.c_void_p(nlos.data_ptr()), sp),
                "kfpos_synth_toa_ranges_nlos")
    else:
        L.check(L.lib().kfpos_synth_toa_ranges(*args, sp), "kfpos_synth_toa_ranges")

    def truth_at(name, times):
        times = np.ascontiguousarray(times, dtype=np.float64)
        tr = buf(name, (len(times), 3, N), torch.float64)
        L.check(L.lib().kfpos_synth_k8_truth(dev.index or 0, N, int(first_filter), C.c_uint64(seed), len(times),
                                             C.c_void_p(times.ctypes.data), float(tag_z), C.c_void_p(tr.data_ptr()),
                                             sp), "kfpos_synth_k8_truth")
        return tr
    res = dict(ranges=ranges, dt=float(period), t=t)
    if want_nlos:
        res["nlos"] = nlos
    if truth is not None:
        if want_truth:
            res["truth"] = truth
        res["truth_end"] = truth[-1]
    elif want_truth:
        res["truth"] = truth_at("truth", t)
        res["truth_end"] = res["truth"][-1]
    else:
        res["truth_end"] = truth_at("truth_end", t[-1:])[0]
    if want_x0:
        x0 = buf("x0", (6, N), torch.float64)
        x0.zero_()
        x0[:3] = truth_at("truth0", [0.0])[0]
        res["x0"] = x0
    return res


def toa_montecarlo(batch, n_epochs, chunk, anchors, seed=SEED, period=0.1, sigma_r=0.10, p_missing=0.0, p_nlos=0.0,
                   nlos_mean=0.8, tag_z=1.0, first_filter=0, fmt=None, err=0.01, epoch0=0, init_state=True,
                   stream=None, hist=None, score=False, *, crlb=None, obstacles=None, walk=None):
    """A Monte Carlo run of any length on a T6 Batch (anchors set to `anchors`), in chunks of `chunk` epochs:
    for each chunk toa_montecarlo_chunk generates the rangings and the truth, Batch.set_truth_traj registers the
    truth (which resets the row cursor, so the chunk's rows start at 0), Batch.replay_toa runs the chunk and
    Batch.epoch_stats reads its rows.  init_state: start from the truth at t = 0 with zero velocity (and the
    batch's initial covariance); False continues from the batch's state at epoch epoch0.  The batch's filter f
    is global filter first_filter + f.  Returns the [n_epochs][6] rows of kfpos_batch_epoch_stats for
    batch.epoch_summary (RMSE(t), ANEES(t)); the truth is unregistered on return.
    hist=(edges, quantity): also a per-epoch histogram (Batch.set_error_hist), read chunk by chunk beside the
    statistics; then returns (rows, counts [n_epochs][len(edges) + 1] uint64), and the histogram is
    unregistered on return as well.
    score=True: each chunk also generates its NLOS mask, the replay writes its selection into a reused device
    buffer and Batch.score_selection scores it; the [n_epochs][8] uint64 scores (batch.selection_summary) are
    appended as the last element of the return value, a tuple then.
    crlb=("present", "los", "used") or any of them: each chunk also calls Batch.crlb for each set with its truth,
    log, NLOS mask and selection, at the generator's ranging variance sigma_r^2 + (1 mm)^2 / 12 (its noise and its
    floor to whole millimetres); a dict {set: [n_epochs][4]} (batch.crlb_summary) is appended as the last element
    of the return value, a tuple then.
    obstacles: the boxes of toa_montecarlo_chunk (DESIGN §4.5f); score and crlb "los" then use the mask that also
    marks the rangings they block.
    walk=dict(accel_sd=..., v_max=..., lo=..., hi=...): the tag follows the random walk of walk_truth_chunk (DESIGN
    §4.5g) instead of the Lissajous, with the run's seed, period and first_filter; tag_z is then unused.  The walk
    starts at epoch0 from its drawn initial state (init_state sets the batch to it, as x0), and its state is carried
    from chunk to chunk on the device, so any chunk length gives the same run."""
    from . import lib as L
    if batch.model != L.MODEL_T6:
        raise ValueError("toa_montecarlo runs T6 batches; ML batches take toa_montecarlo_chunk output directly")
    if int(chunk) <= 0 or int(n_epochs) <= 0:
        raise ValueError("toa_montecarlo: n_epochs and chunk must be positive")
    kw = dict(seed=seed, period=period, sigma_r=sigma_r, p_missing=p_missing, p_nlos=p_nlos, nlos_mean=nlos_mean,
              tag_z=tag_z, first_filter=first_filter, fmt=fmt, stream=stream, obstacles=obstacles)
    crlb = (crlb,) if isinstance(crlb, str) else tuple(crlb or ())
    bounds = {name: [] for name in crlb}
    want_sel, want_nlos = score or "used" in crlb, score or "los" in crlb
    var = float(sigma_r) ** 2 + 1e-6 / 12.0
    rows, counts, scores, bufs, wbufs = [], [], [], {}, {}
    sel = wstate = None
    if walk is not None:
        walk = dict(walk)
        if set(walk) != {"accel_sd", "v_max", "lo", "hi"}:
            raise ValueError("toa_montecarlo: walk takes exactly accel_sd, v_max, lo and hi")
    if hist is not None:
        batch.set_error_hist(hist[0], hist[1])
    try:
        for k0 in range(0, int(n_epochs), int(chunk)):
            n = min(int(chunk), int(n_epochs) - k0)
            x0 = None
            if walk is None:
                w = toa_montecarlo_chunk(batch.N, epoch0 + k0, n, anchors, "cuda:%d" % batch.device, want_truth=True,
                                         want_x0=init_state and k0 == 0, out=bufs, want_nlos=want_nlos, **kw)
                x0 = w.get("x0")
            else:
                wk = walk_truth_chunk(batch.N, epoch0 + k0, n, "cuda:%d" % batch.device, seed=seed, period=period,
                                      first_filter=first_filter, state=wstate, want_x0=init_state and k0 == 0,
                                      out=wbufs, stream=stream, **walk)
                wstate, x0 = wk["state"], wk.get("x0")
                w = toa_montecarlo_chunk(batch.N, epoch0 + k0, n, anchors, "cuda:%d" % batch.device, want_truth=True,
                                         out=bufs, want_nlos=want_nlos, truth=wk["truth"], **kw)
            if init_state and k0 == 0:
                batch.set_state(x0, None, stream=stream)
            batch.set_truth_traj(w["truth"], stream=stream)
            if want_sel and (sel is None or sel.shape[0] != n):
                import torch
                sel = torch.empty((n, batch.N), dtype=torch.int32, device="cuda:%d" % batch.device)
            batch.replay_toa(w["dt"], w["ranges"], err=err, sel=sel, stream=stream)
            rows.append(batch.epoch_stats(stream=stream))
            if hist is not None:
                counts.append(batch.error_hist(stream=stream))
            if score:
                scores.append(batch.score_selection(w["ranges"], sel, w["nlos"], stream=stream))
            for name in crlb:
                bounds[name].append(batch.crlb(w["truth"], w["ranges"], var, sel, w.get("nlos"), set=name,
                                               stream=stream))
    finally:
        batch.set_truth_traj(None, stream=stream)
        if hist is not None:
            batch.set_error_hist(None)
    out = (np.concatenate(rows, axis=0),)
    if hist is not None:
        out += (np.concatenate(counts, axis=0),)
    if score:
        out += (np.concatenate(scores, axis=0),)
    if crlb:
        out += ({name: np.concatenate(b, axis=0) for name, b in bounds.items()},)
    return out if len(out) > 1 else out[0]
