"""Python host side of the C ABI: a `Batch` of N independent filters on one GPU.

Arrays may be numpy arrays (host: the library stages them) or CUDA torch tensors
(device: passed through untouched).  torch is only used for device memory and
streams; all arithmetic happens inside libkfpos_b200.so.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional

import numpy as np

from . import lib as L

_FMT_NP = {np.dtype(np.float64): L.FMT_F64_M, np.dtype(np.int32): L.FMT_I32_MM,
           np.dtype(np.uint16): L.FMT_U16_MM}


def _is_torch(a) -> bool:
    return type(a).__module__.startswith("torch")


def _ptr(a, dtype=None):
    """(void* address, keep-alive object) of a numpy array / torch tensor / None."""
    if a is None:
        return None, None
    if _is_torch(a):
        if not a.is_contiguous():
            raise ValueError("tensor arguments must be contiguous")
        return C.c_void_p(a.data_ptr()), a
    arr = np.ascontiguousarray(a, dtype=dtype)
    return C.c_void_p(arr.ctypes.data), arr


def _fmt_of(a) -> int:
    if _is_torch(a):
        import torch
        return {torch.float64: L.FMT_F64_M, torch.int32: L.FMT_I32_MM, torch.uint16: L.FMT_U16_MM,
                torch.int16: L.FMT_U16_MM}[a.dtype]
    return _FMT_NP[np.asarray(a).dtype]


def _stream_ptr(stream) -> Optional[C.c_void_p]:
    if stream is None:
        return None
    return C.c_void_p(int(getattr(stream, "cuda_stream", stream)))


def _comm_ptr(comm) -> Optional[C.c_void_p]:
    """A raw ncclComm_t (an int or c_void_p, see shard.nccl_comm) as the library takes it; None = no communicator."""
    return C.c_void_p(int(comm)) if comm else None


def make_config(**kw) -> L.KfposConfig:
    cfg = L.KfposConfig()
    L.lib().kfpos_config_default(C.byref(cfg))
    xml = kw.pop("xml", None)
    for blob in ([xml] if isinstance(xml, (str, bytes)) else (xml or [])):
        data = blob.encode() if isinstance(blob, str) else blob
        L.check(L.lib().kfpos_config_load_xml(C.byref(cfg), data), "kfpos_config_load_xml")
    for k, v in kw.items():
        if k == "ml_start":
            for i in range(3):
                cfg.ml_start[i] = float(v[i])
        else:
            if not hasattr(cfg, k):
                raise AttributeError(f"kfpos_config has no field {k!r}")
            setattr(cfg, k, v)
    return cfg


class Batch:
    """N identical-configuration filters (or ML epoch slots) on one GPU."""

    def __init__(self, model: int, n_filters: int, config: Optional[L.KfposConfig] = None,
                 device: int = 0, anchors=None, **cfg_kw):
        self._h = C.c_void_p()
        self.cfg = config if config is not None else make_config(**cfg_kw)
        self.model = model
        self.N = int(n_filters)
        self.device = int(device)
        L.check(L.lib().kfpos_batch_create(C.byref(self._h), int(device), int(model),
                                           C.c_int64(self.N), C.byref(self.cfg)), "kfpos_batch_create")
        self.n = L.lib().kfpos_batch_state_dim(self._h)
        self.n_anchors = 0
        if anchors is not None:
            self.set_anchors(anchors)

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            L.lib().kfpos_batch_destroy(self._h)
            self._h = C.c_void_p()

    __del__ = close

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    # ------------------------------------------------------------------ setup
    def set_anchors(self, xyz):
        xyz = np.ascontiguousarray(xyz, dtype=np.float64).reshape(-1, 3)
        L.check(L.lib().kfpos_batch_set_anchors(self._h, len(xyz), C.c_void_p(xyz.ctypes.data)),
                "kfpos_batch_set_anchors")
        self.n_anchors = len(xyz)

    def set_state(self, x, P=None, stream=None):
        """x: [n][N] (rows beyond those given are zero if x has fewer rows); P [n*n][N] or None."""
        if not _is_torch(x):
            x = np.asarray(x, dtype=np.float64).reshape(-1, self.N)
            if x.shape[0] < self.n:
                x = np.vstack([x, np.zeros((self.n - x.shape[0], self.N))])
        px, kx = _ptr(x, np.float64)
        pP, kP = _ptr(P, np.float64)
        L.check(L.lib().kfpos_batch_set_state(self._h, px, pP, _stream_ptr(stream)), "kfpos_batch_set_state")

    def get_state(self, want_P=True, stream=None):
        x = np.empty((self.n, self.N))
        P = np.empty((self.n * self.n, self.N)) if want_P else None
        st = np.empty(self.N, dtype=np.int32)
        L.check(L.lib().kfpos_batch_get_state(self._h, C.c_void_p(x.ctypes.data),
                                              C.c_void_p(P.ctypes.data) if want_P else None,
                                              C.c_void_p(st.ctypes.data), _stream_ptr(stream)),
                "kfpos_batch_get_state")
        return x, P, st

    def get_latches(self, stream=None):
        """The latched sensor members of a running K8 / T9 batch: (latch [16][N], has [N], latch_u [16])."""
        latch = np.empty((16, self.N)); has = np.empty(self.N, dtype=np.int32); u = np.empty(16)
        L.check(L.lib().kfpos_batch_get_latches(self._h, C.c_void_p(latch.ctypes.data), C.c_void_p(has.ctypes.data),
                                                C.c_void_p(u.ctypes.data), _stream_ptr(stream)), "kfpos_batch_get_latches")
        return latch, has, u

    def set_latches(self, latch, has, latch_u, stream=None):
        a = [np.ascontiguousarray(latch, dtype=np.float64), np.ascontiguousarray(has, dtype=np.int32),
             np.ascontiguousarray(latch_u, dtype=np.float64)]
        L.check(L.lib().kfpos_batch_set_latches(self._h, C.c_void_p(a[0].ctypes.data), C.c_void_p(a[1].ctypes.data),
                                                C.c_void_p(a[2].ctypes.data), _stream_ptr(stream)), "kfpos_batch_set_latches")

    def get_state_into(self, x=None, P=None, status=None, stream=None):
        """Device-to-device variant of get_state for torch tensors."""
        L.check(L.lib().kfpos_batch_get_state(self._h, _ptr(x)[0], _ptr(P)[0], _ptr(status)[0],
                                              _stream_ptr(stream)), "kfpos_batch_get_state")

    # ------------------------------------------------------------------ steps
    def _err(self, err):
        if err is None or np.isscalar(err):
            return float(0.0 if err is None else err), None, None
        p, keep = _ptr(err, np.float64)
        return 0.0, p, keep

    def step_toa(self, dt, ranges, err=0.01, stream=None):
        es, ep, keep = self._err(err)
        pr, kr = _ptr(ranges)
        L.check(L.lib().kfpos_batch_step_toa(self._h, float(dt), pr, _fmt_of(ranges), es, ep,
                                             _stream_ptr(stream)), "kfpos_batch_step_toa")

    def replay_toa(self, dt, ranges, err=0.01, traj=None, sel=None, want_traj=False, want_sel=False,
                   stream=None):
        """ranges [T][M][N]; dt scalar or [T].  Returns (traj, sel) (numpy, or the tensors given)."""
        T = int(ranges.shape[0])
        dts = np.ascontiguousarray(np.broadcast_to(np.asarray(dt, dtype=np.float64), (T,)))
        es, ep, keep = self._err(err)
        pr, kr = _ptr(ranges)
        if traj is None and want_traj:
            traj = np.empty((T, 3, self.N))
        if sel is None and want_sel:
            sel = np.empty((T, self.N), dtype=np.int32)
        L.check(L.lib().kfpos_batch_replay_toa(self._h, T, C.c_void_p(dts.ctypes.data), pr,
                                               _fmt_of(ranges), es, ep, _ptr(traj)[0], _ptr(sel)[0],
                                               _stream_ptr(stream)), "kfpos_batch_replay_toa")
        return traj, sel

    def replay_epochs(self, dt_per_filter, ranges, err=0.01, traj=None, want_traj=False, stream=None):
        """T6 / K8 / T9: ranges [T][M][N] with per-filter time steps dt_per_filter [T][N] (< 0 = no
        epoch), the output of assemble_epochs()."""
        T = int(ranges.shape[0])
        es, ep, keep = self._err(err)
        pr, kr = _ptr(ranges)
        pd, kd = _ptr(dt_per_filter, np.float64)
        if traj is None and want_traj:
            traj = np.empty((T, 3, self.N))
        L.check(L.lib().kfpos_batch_replay_epochs(self._h, T, pd, pr, _fmt_of(ranges), es, ep, _ptr(traj)[0],
                                                  _stream_ptr(stream)), "kfpos_batch_replay_epochs")
        return traj

    def step_px4(self, dt, ix, iy, irz, itime_us, quality, stream=None):
        a = [_ptr(v, np.float64) for v in (ix, iy, irz, itime_us)]
        q = _ptr(quality, np.int32)
        L.check(L.lib().kfpos_batch_step_px4(self._h, float(dt), a[0][0], a[1][0], a[2][0], a[3][0], q[0],
                                             _stream_ptr(stream)), "kfpos_batch_step_px4")

    def step_imu(self, dt, ang_vel, lin_acc, cov_ang_vel=None, cov_acc=None, stream=None):
        """ang_vel, lin_acc: [3][N]; cov_*: 9 doubles (row-major 3x3) for the whole batch or None."""
        a = [_ptr(v, np.float64) for v in (ang_vel, lin_acc)]
        c = [None if v is None else np.ascontiguousarray(v, dtype=np.float64).reshape(9) for v in (cov_ang_vel, cov_acc)]
        cp = [None if v is None else C.c_void_p(v.ctypes.data) for v in c]
        L.check(L.lib().kfpos_batch_step_imu(self._h, float(dt), a[0][0], cp[0], a[1][0], cp[1],
                                             _stream_ptr(stream)), "kfpos_batch_step_imu")

    def replay_events(self, events, ranges=None, sensors=None, err=0.01, traj=None, want_traj=False, stream=None,
                      dt_per_filter=None):
        """events: list of (kind, dt, offset_row[, aux]) ; ranges [T][M][N] (or [rows][N]); sensors [R][N] f64.
        dt_per_filter [n_events][N]: per-filter time steps (< 0 = the filter has no such event), the ragged replay
        of schedules merged by merge_streams (kfpos_batch_replay_events_ragged)."""
        n = len(events)
        arr = (L.KfposEvent * n)()
        n_toa = 0
        for i, ev in enumerate(events):
            arr[i].kind, arr[i].dt, arr[i].offset = int(ev[0]), float(ev[1]), int(ev[2])
            if len(ev) > 3 and ev[3] is not None:
                for k, v in enumerate(ev[3]):
                    arr[i].aux[k] = float(v)
            n_toa += ev[0] == L.EV_TOA
        es, ep, keep = self._err(err)
        pr, kr = _ptr(ranges)
        ps, ks = _ptr(sensors, np.float64)
        srows = 0 if sensors is None else int(np.prod(sensors.shape[:-1]))
        if traj is None and want_traj:
            traj = np.empty((n_toa, 3, self.N))
        fmt = _fmt_of(ranges) if ranges is not None else L.FMT_F64_M
        if dt_per_filter is not None:
            pd, kd = _ptr(dt_per_filter, np.float64)
            L.check(L.lib().kfpos_batch_replay_events_ragged(self._h, n, C.cast(arr, C.c_void_p), pd, pr, fmt, es, ep, ps,
                                                             C.c_int64(srows), _ptr(traj)[0], _stream_ptr(stream)),
                    "kfpos_batch_replay_events_ragged")
            return traj
        L.check(L.lib().kfpos_batch_replay_events(self._h, n, C.cast(arr, C.c_void_p), pr, fmt, es, ep, ps,
                                                  C.c_int64(srows), _ptr(traj)[0], _stream_ptr(stream)),
                "kfpos_batch_replay_events")
        return traj

    def step_mag(self, dt, mag, stream=None):
        p, k = _ptr(mag, np.float64)
        L.check(L.lib().kfpos_batch_step_mag(self._h, float(dt), p, _stream_ptr(stream)), "kfpos_batch_step_mag")

    def step_compass(self, dt, compass, stream=None):
        p, k = _ptr(compass, np.float64)
        L.check(L.lib().kfpos_batch_step_compass(self._h, float(dt), p, _stream_ptr(stream)),
                "kfpos_batch_step_compass")

    def get_pose(self, dt, stream=None):
        x = np.empty((self.n, self.N))
        P = np.empty((self.n * self.n, self.N))
        L.check(L.lib().kfpos_batch_get_pose(self._h, float(dt), C.c_void_p(x.ctypes.data),
                                             C.c_void_p(P.ctypes.data), _stream_ptr(stream)),
                "kfpos_batch_get_pose")
        return x, P

    def get_pose_msg(self, dt, stream=None):
        """getPose in the publisher's layout: (pose [13][N], cov [36][N])."""
        pose = np.empty((13, self.N))
        cov = np.empty((36, self.N))
        L.check(L.lib().kfpos_batch_get_pose_msg(self._h, float(dt), C.c_void_p(pose.ctypes.data),
                                                 C.c_void_p(cov.ctypes.data), _stream_ptr(stream)),
                "kfpos_batch_get_pose_msg")
        return pose, cov

    # --------------------------------------------------------------------- ML
    def ml_solve(self, ranges, err=0.01, out=None, stream=None):
        """ranges [M][N].  Returns dict(pos [3][N], cov [9][N], iters, sel [2][N], status)."""
        es, ep, keep = self._err(err)
        pr, kr = _ptr(ranges)
        if out is None:
            out = dict(pos=np.empty((3, self.N)), cov=np.empty((9, self.N)),
                       iters=np.empty(self.N, dtype=np.int32), sel=np.empty((2, self.N), dtype=np.int32),
                       status=np.empty(self.N, dtype=np.int32))
        L.check(L.lib().kfpos_batch_ml_solve(self._h, pr, _fmt_of(ranges), es, ep,
                                             _ptr(out.get("pos"))[0], _ptr(out.get("cov"))[0],
                                             _ptr(out.get("iters"))[0], _ptr(out.get("sel"))[0],
                                             _ptr(out.get("status"))[0], _stream_ptr(stream)),
                "kfpos_batch_ml_solve")
        return out

    def _result(self, out, readback, shape, counts=False):
        """The array a reader fills: `out` when given, else zeros on the host when `readback`, else a new device
        tensor on this batch's GPU.  float64, or for counts uint64 on the host and int64 on the device."""
        if out is not None:
            return out
        if readback:
            return np.zeros(shape, dtype=np.uint64 if counts else np.float64)
        import torch
        return torch.empty(shape, dtype=torch.int64 if counts else torch.float64, device="cuda:%d" % self.device)

    # ------------------------------------------------------------ diagnostics
    def counters(self, reset=False, stream=None):
        buf = (C.c_double * 8)()
        L.check(L.lib().kfpos_batch_get_counters(self._h, C.byref(buf), int(reset), _stream_ptr(stream)),
                "kfpos_batch_get_counters")
        v = list(buf)
        return dict(updates=v[0], ml_iters=v[1], cost_evals=v[2], gain_evals=v[3], bad=v[4], ignored=v[5],
                    ml_capped=v[6], ml_cycles=v[7])

    def set_truth(self, truth, stream=None):
        """Registers the ground truth SoA [3][N]: replay launches then end with the block-level reduction of the
        error statistics (kfpos_batch_set_truth).  A device tensor is borrowed -- keep it alive."""
        p, k = _ptr(truth, np.float64)
        self._truth_keep = k
        L.check(L.lib().kfpos_batch_set_truth(self._h, p, _stream_ptr(stream)), "kfpos_batch_set_truth")

    def error_stats(self, truth=None, stream=None, readback=True):
        """[sum |e|^2, sum |e_xy|^2, n, n_bad]; truth None = the registered one; readback False = enqueue only
        (the result stays on the device for stats_allreduce, no host synchronisation)."""
        buf = (C.c_double * 4)()
        p, k = _ptr(truth, np.float64)
        L.check(L.lib().kfpos_batch_error_stats(self._h, p, C.byref(buf) if readback else None, _stream_ptr(stream)),
                "kfpos_batch_error_stats")
        return np.array(list(buf)) if readback else None

    def stats_allreduce(self, comm=None, truth=None, stream=None):
        """kfpos_stats_allreduce: the statistics of the batches of all ranks of the NCCL communicator `comm`
        (a raw ncclComm_t as an int / c_void_p, see shard.nccl_comm; None = this batch alone).
        Returns [sum |e|^2, sum |e_xy|^2, n, n_bad, rmse, rmse_xy]."""
        buf = (C.c_double * 6)()
        p, k = _ptr(truth, np.float64)
        L.check(L.lib().kfpos_stats_allreduce(self._h, _comm_ptr(comm), p, C.byref(buf), _stream_ptr(stream)),
                "kfpos_stats_allreduce")
        return np.array(list(buf))

    # ------------------------------------------------- per-epoch statistics
    def set_truth_traj(self, truth, stream=None):
        """Registers the truth trajectory SoA [rows][3][N] (K8: z = the tag height) for the per-epoch statistics:
        every replay launch then leaves the partial sums of its output rows and advances the row cursor
        (kfpos_batch_set_truth_traj; set_state resets the cursor).  A device tensor is borrowed -- keep it alive.
        None unregisters."""
        rows = 0 if truth is None else int(truth.shape[0])
        p, k = _ptr(truth, np.float64)
        self._etruth_keep = k
        self._es_rows = rows
        L.check(L.lib().kfpos_batch_set_truth_traj(self._h, C.c_int64(rows), p, _stream_ptr(stream)),
                "kfpos_batch_set_truth_traj")

    def epoch_stats(self, readback=True, out=None, stream=None):
        """[rows][6] per output row: sum |e|^2, sum |e_xy|^2, n, n with status != 0 in that epoch, sum NEES,
        n in the NEES (kfpos_batch_epoch_stats).  out: a device tensor [rows][6] to fill asynchronously
        (returned as given); readback False without `out`: a new device tensor, filled asynchronously."""
        rows = getattr(self, "_es_rows", 0)
        out = self._result(out, readback, (rows, 6))
        L.check(L.lib().kfpos_batch_epoch_stats(self._h, C.c_int64(rows), _ptr(out)[0], _stream_ptr(stream)),
                "kfpos_batch_epoch_stats")
        return out

    def epoch_stats_allreduce(self, comm=None, stream=None):
        """kfpos_epoch_stats_allreduce: epoch_stats summed over the ranks of the NCCL communicator `comm` (a raw
        ncclComm_t as an int / c_void_p, see shard.nccl_comm; None = this batch alone).  Returns [rows][6]."""
        rows = getattr(self, "_es_rows", 0)
        out = np.zeros((rows, 6))
        L.check(L.lib().kfpos_epoch_stats_allreduce(self._h, _comm_ptr(comm), C.c_int64(rows),
                                                    C.c_void_p(out.ctypes.data), _stream_ptr(stream)),
                "kfpos_epoch_stats_allreduce")
        return out

    # ------------------------------------------------ per-epoch error histograms
    _HIST_QUANTITY = {"err": L.HIST_ERR, "err_xy": L.HIST_ERR_XY, "nees": L.HIST_NEES}

    def set_error_hist(self, edges, quantity="err"):
        """Registers a per-epoch histogram of `quantity` ("err" = |p - truth| in m, "err_xy" = the x-y error in m,
        "nees") with the bin edges `edges` (1..255 finite, strictly increasing values; >= 0 for the errors):
        bin k of a row counts the filters with exactly k edges <= their value (kfpos_batch_set_error_hist).  It
        is filled while a truth trajectory is registered (set_truth_traj) and survives its re-registration.
        None (or no edges) unregisters."""
        if quantity not in self._HIST_QUANTITY:
            raise ValueError(f"set_error_hist: quantity must be one of {sorted(self._HIST_QUANTITY)}")
        e = None if edges is None else np.ascontiguousarray(edges, dtype=np.float64).reshape(-1)
        n = 0 if e is None else len(e)
        L.check(L.lib().kfpos_batch_set_error_hist(self._h, self._HIST_QUANTITY[quantity], n,
                                                   C.c_void_p(e.ctypes.data) if n else None),
                "kfpos_batch_set_error_hist")
        self._eh_bins = n + 1 if n else 0

    def error_hist(self, readback=True, out=None, stream=None):
        """[rows][n_edges + 1] uint64 counts per output row (kfpos_batch_error_hist).  out: a device tensor
        (int64 or uint64) of that shape to fill asynchronously (returned as given); readback False without
        `out`: a new device int64 tensor, filled asynchronously."""
        rows, bins = getattr(self, "_es_rows", 0), getattr(self, "_eh_bins", 0)
        out = self._result(out, readback, (rows, bins), counts=True)
        L.check(L.lib().kfpos_batch_error_hist(self._h, C.c_int64(rows), _ptr(out)[0], _stream_ptr(stream)),
                "kfpos_batch_error_hist")
        return out

    def error_hist_allreduce(self, comm=None, stream=None):
        """kfpos_error_hist_allreduce: error_hist summed over the ranks of the NCCL communicator `comm` (a raw
        ncclComm_t as an int / c_void_p, see shard.nccl_comm; None = this batch alone).  Exact for any shard
        sizes.  Returns [rows][n_edges + 1] uint64."""
        rows, bins = getattr(self, "_es_rows", 0), getattr(self, "_eh_bins", 0)
        out = np.zeros((rows, bins), dtype=np.uint64)
        L.check(L.lib().kfpos_error_hist_allreduce(self._h, _comm_ptr(comm), C.c_int64(rows),
                                                   C.c_void_p(out.ctypes.data), _stream_ptr(stream)),
                "kfpos_error_hist_allreduce")
        return out

    # ------------------------------------------------------- selection scores
    def score_selection(self, ranges, sel=None, nlos=None, out=None, readback=True, stream=None):
        """NLOS detection scores of the selection this batch just made (kfpos_batch_score_selection): T6 ranges
        [T][M][N] with the `sel` [T][N] of replay_toa; ML ranges [M][N] with the `sel` [2][N] of ml_solve.  nlos:
        the [rows][N] masks of synth.toa_montecarlo_chunk(want_nlos=True) (int32 holding the uint32 bits), or None
        (no ranging is NLOS).  sel may be None where the configuration drops nothing (plain T6, ML variant 0).
        Returns counts [rows][8] (columns in selection_summary) as uint64 numpy; out: a device tensor (int64 or
        uint64) of that shape to fill asynchronously (returned as given); readback False without `out`: a new
        device int64 tensor, filled asynchronously."""
        rows = 1 if self.model == L.MODEL_ML else int(ranges.shape[0])
        out = self._result(out, readback, (rows, L.SCORE_COLS), counts=True)
        pr, kr = _ptr(ranges)
        ps, ks = _ptr(sel, np.int32)
        pn, kn = _ptr(nlos, np.uint32)
        L.check(L.lib().kfpos_batch_score_selection(self._h, rows, pr, _fmt_of(ranges), ps, pn, _ptr(out)[0],
                                                    _stream_ptr(stream)), "kfpos_batch_score_selection")
        return out

    # ------------------------------------------------------- Cramer-Rao bound
    _CRLB_SET = {"present": L.CRLB_PRESENT, "los": L.CRLB_LOS, "used": L.CRLB_USED}

    def crlb(self, truth, ranges, var, sel=None, nlos=None, set="present", out=None, readback=True, stream=None):
        """Per-epoch Cramer-Rao bound of the position (kfpos_batch_crlb) for the rangings of each filter in the set
        `set`: "present" (in the log), "los" (present and not NLOS in `nlos`) or "used" (kept by this batch's
        selection `sel`, read as score_selection reads it).  T6 / K8 / T9: truth [T][3][N], ranges [T][M][N], sel
        [T][N] of replay_toa; ML: truth [3][N], ranges [M][N], sel [2][N] of ml_solve.  var: the true ranging
        variance in m^2, a scalar or [rows][M][N].  nlos: the masks of synth.toa_montecarlo_chunk(want_nlos=True).
        Returns [rows][4] sums over the filters (columns in crlb_summary) as float64 numpy; out: a device tensor of
        that shape to fill asynchronously (returned as given); readback False without `out`: a new device tensor,
        filled asynchronously."""
        if set not in self._CRLB_SET:
            raise ValueError(f"crlb: set must be one of {sorted(self._CRLB_SET)}")
        rows = 1 if self.model == L.MODEL_ML else int(ranges.shape[0])
        out = self._result(out, readback, (rows, L.CRLB_COLS))
        vs, pv, kv = (float(var), None, None) if np.isscalar(var) else (0.0, *_ptr(var, np.float64))
        pt, kt = _ptr(truth, np.float64)
        pr, kr = _ptr(ranges)
        ps, ks = _ptr(sel, np.int32)
        pn, kn = _ptr(nlos, np.uint32)
        L.check(L.lib().kfpos_batch_crlb(self._h, self._CRLB_SET[set], rows, pt, pr, _fmt_of(ranges), vs, pv, ps, pn,
                                         _ptr(out)[0], _stream_ptr(stream)), "kfpos_batch_crlb")
        return out


def epoch_summary(stats):
    """Per-row summary of epoch_stats / epoch_stats_allreduce output [rows][6]: dict of arrays rmse, rmse_xy
    (over the filters with a finite error), anees (average NEES over the filters it counts), n, n_bad.
    Rows without filters give NaN."""
    s = np.asarray(stats, dtype=np.float64).reshape(-1, 6)
    with np.errstate(invalid="ignore", divide="ignore"):
        n = s[:, 2]
        ne = s[:, 5]
        return dict(rmse=np.where(n > 0, np.sqrt(s[:, 0] / n), np.nan),
                    rmse_xy=np.where(n > 0, np.sqrt(s[:, 1] / n), np.nan),
                    anees=np.where(ne > 0, s[:, 4] / ne, np.nan), n=n.copy(), n_bad=s[:, 3].copy())


def selection_summary(counts, n_filters):
    """Per-row rates of score_selection output counts [rows][8] over a batch of n_filters filters (the sum of the
    shards' sizes for summed counts): detection = NLOS rangings dropped / NLOS rangings present; false_drop = LOS
    rangings dropped / LOS rangings present; clean = filters with an NLOS ranging whose used set has none / filters
    with an NLOS ranging; false_alarm = filters without an NLOS ranging that dropped one / filters without an NLOS
    ranging.  A zero denominator gives NaN."""
    c = np.asarray(counts).astype(np.float64).reshape(-1, 8)

    def rate(num, den):
        with np.errstate(invalid="ignore", divide="ignore"):
            return np.where(den > 0, num / np.where(den > 0, den, 1.0), np.nan)
    return dict(detection=rate(c[:, 3], c[:, 2]), false_drop=rate(c[:, 1] - c[:, 3], c[:, 0] - c[:, 2]),
                clean=rate(c[:, 5], c[:, 4]), false_alarm=rate(c[:, 7], float(n_filters) - c[:, 4]))


def crlb_summary(rows):
    """Per-row summary of crlb output [rows][4]: dict of arrays rmse_bound = sqrt(mean tr J^-1) and rmse_xy_bound
    (the RMS position-error floors over the filters with a bound, to set beside epoch_summary's rmse and
    rmse_xy), n (filters with a bound) and n_none (filters without).  Rows without a bound give NaN."""
    c = np.asarray(rows, dtype=np.float64).reshape(-1, 4)
    with np.errstate(invalid="ignore", divide="ignore"):
        n = c[:, 2]
        return dict(rmse_bound=np.where(n > 0, np.sqrt(c[:, 0] / n), np.nan),
                    rmse_xy_bound=np.where(n > 0, np.sqrt(c[:, 1] / n), np.nan), n=n.copy(), n_none=c[:, 3].copy())


def rank_tree(rows_per_rank):
    """The rows of the ranks of a sharded run ([n_ranks][rows][W], rank order: e.g. torch.distributed.all_gather of
    each rank's crlb output) added by the pairwise tree over the rank index, level by level a[i] += a[i + stride]
    -- the adds of the library's error_stats_tree, in its order.  With aligned power-of-two shards (multiples of
    32 filters) the result equals the whole batch's rows bit for bit.  Returns [rows][W]."""
    a = np.array(rows_per_rank, dtype=np.float64)
    if a.ndim < 2 or a.shape[0] == 0:
        raise ValueError("rank_tree: expects [n_ranks][rows][W] with at least one rank")
    stride = 1
    while stride < a.shape[0]:
        i = np.arange(0, a.shape[0] - stride, 2 * stride)
        a[i] = a[i] + a[i + stride]
        stride *= 2
    return a[0]


def hist_quantiles(counts, edges, q):
    """Brackets quantiles of each row of error_hist output counts [rows][n_edges + 1] with the edges it was
    registered with.  For each row and each q in `q` (in [0, 1]) returns the interval [lo, hi) of the bin that
    holds the q-quantile: the smallest value v with at least max(1, ceil(q * n)) of the row's n values <= v.
    The quantile is only bracketed, not interpolated inside its bin, so it is known to one bin width.  lo of
    bin 0 is 0 (errors and NEES are never negative); hi of the last bin is inf.  Empty rows give NaN.
    Returns (lo, hi), each [rows][len(q)]."""
    c = np.asarray(counts).astype(np.float64)
    c = c.reshape(-1, c.shape[-1])
    e = np.asarray(edges, dtype=np.float64).reshape(-1)
    if c.shape[1] != len(e) + 1:
        raise ValueError("hist_quantiles: counts must have len(edges) + 1 bins")
    qs = np.atleast_1d(np.asarray(q, dtype=np.float64))
    if np.any(qs < 0) or np.any(qs > 1):
        raise ValueError("hist_quantiles: q must lie in [0, 1]")
    cum = np.cumsum(c, axis=1)
    n = cum[:, -1]
    # the bin of the k-th smallest value: the first bin whose cumulative count reaches k
    k = np.maximum(1.0, np.ceil(qs[None, :] * n[:, None]))
    b = np.minimum((cum[:, :, None] < k[:, None, :]).sum(axis=1), c.shape[1] - 1)
    lo = np.concatenate([[0.0], e])[b]
    hi = np.concatenate([e, [np.inf]])[b]
    lo[n <= 0] = np.nan
    hi[n <= 0] = np.nan
    return lo, hi


def assemble_epochs(anchor, seq, range_mm, t, n_anchors, max_epochs, err=None, fix_row_clear=False, first_dt=0.1,
                    device=0, out=None, stream=None):
    """Ranging aggregation of PosGenerator for N logs of L messages (SoA [L][N]; numpy or CUDA torch
    tensors: uint8 anchor index, uint8 seq, int32 range_mm, f64 arrival time, optional f64 err).
    Returns dict(ranges int32 [T][M][N], err [T][M][N] or None, dt [T][N], n_epochs [N], t [T][N] = the report
    times); `out` may supply device tensors under the same keys."""
    Lm, N = int(anchor.shape[0]), int(anchor.shape[1])
    M, T = int(n_anchors), int(max_epochs)
    if out is None:
        out = dict(ranges=np.empty((T, M, N), dtype=np.int32), err=None if err is None else np.empty((T, M, N)),
                   dt=np.empty((T, N)), n_epochs=np.empty(N, dtype=np.int32), t=np.empty((T, N)))
    keep = [_ptr(anchor, np.uint8), _ptr(seq, np.uint8), _ptr(range_mm, np.int32), _ptr(err, np.float64),
            _ptr(t, np.float64)]
    L.check(L.lib().kfpos_assemble_epochs_t(int(device), N, Lm, M, keep[0][0], keep[1][0], keep[2][0], keep[3][0],
                                            keep[4][0], T, L.ASM_FIX_ROW_CLEAR if fix_row_clear else 0, float(first_dt),
                                            _ptr(out["ranges"])[0], _ptr(out.get("err"))[0], _ptr(out["dt"])[0],
                                            _ptr(out.get("n_epochs"))[0], _ptr(out.get("t"))[0], _stream_ptr(stream)),
            "kfpos_assemble_epochs_t")
    return out


def merge_streams(t_epoch, ranges, err, sensors, slot_kind, first_dt=0.1, imu_aux=None, device=0, stream=None):
    """kfpos_merge_streams: N tags' ranging reports (t_epoch [T][N], ranges int32 [T][M][N], err [T][M][N] or None:
    the assembler's outputs) and sensor samples (sensors = {EV kind: (t [L][N], payload [L][rows][N])}) in arrival
    order, laid onto the common schedule `slot_kind` (list of EV kinds).  numpy arrays in, numpy arrays out:
    dict(events = list for Batch.replay_events, dt [S][N], ranges int32 [rows][N], err, sensors [rows][N], n_dropped)."""
    ranges = np.ascontiguousarray(ranges, dtype=np.int32)
    T, M, N = ranges.shape
    t_epoch = np.ascontiguousarray(t_epoch, dtype=np.float64)
    err = None if err is None else np.ascontiguousarray(err, dtype=np.float64)
    sk = np.ascontiguousarray(slot_kind, dtype=np.int32)
    S = len(sk)
    n_toa = int((sk == L.EV_TOA).sum())
    srows = int(sum(L.EV_ROWS[int(k)] for k in sk if k != L.EV_TOA))
    ns = (C.c_int64 * 4)(0, 0, 0, 0)
    tp = (C.c_void_p * 4)()
    pp = (C.c_void_p * 4)()
    keep = []
    for k, (tk, pk) in sensors.items():
        tk = np.ascontiguousarray(tk, dtype=np.float64)
        pk = np.ascontiguousarray(pk, dtype=np.float64)
        assert pk.shape == (tk.shape[0], L.EV_ROWS[k], N)
        keep += [tk, pk]
        ns[k - 1] = tk.shape[0]
        tp[k - 1] = tk.ctypes.data
        pp[k - 1] = pk.ctypes.data
    aux = None if imu_aux is None else np.ascontiguousarray(list(imu_aux) + [0.0] * (9 - len(imu_aux)), dtype=np.float64)
    ev = (L.KfposEvent * S)()
    out = dict(dt=np.empty((S, N)), ranges=np.empty((max(n_toa * M, 1), N), dtype=np.int32),
               err=None if err is None else np.empty((max(n_toa * M, 1), N)), sensors=np.empty((max(srows, 1), N)),
               n_dropped=np.empty(N, dtype=np.int32))
    vp = lambda a: None if a is None else C.c_void_p(a.ctypes.data)
    L.check(L.lib().kfpos_merge_streams(int(device), N, M, T, vp(t_epoch), vp(ranges), vp(err), C.cast(ns, C.c_void_p),
                                        C.cast(tp, C.c_void_p), C.cast(pp, C.c_void_p), S, vp(sk),
                                        float(first_dt), vp(aux), C.cast(ev, C.c_void_p), vp(out["dt"]), vp(out["ranges"]),
                                        vp(out["err"]), vp(out["sensors"]), vp(out["n_dropped"]), _stream_ptr(stream)),
            "kfpos_merge_streams")
    out["events"] = [(int(e.kind), 0.0, int(e.offset), list(e.aux) if e.kind == L.EV_IMU else None) for e in ev]
    return out
