"""GPU: per-epoch error and NEES histograms (kfpos_batch_set_error_hist / kfpos_batch_error_hist) fused into the
T6, K8 and T9 replay kernels -- every count against the host binning of the trajectory (exact) or of the numpy
NEES, row totals against kfpos_batch_epoch_stats, ragged epochs, non-interference, chunking and re-runs,
sharding, the allreduce and the error paths."""
import ctypes as C
import os
import socket
import subprocess
import sys
import textwrap

import numpy as np
import pytest

from roskfpos_b200 import synth

pytestmark = pytest.mark.gpu

INVALID, NOT_READY = -1, -4
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EDGES = np.arange(1, 61) * 0.01           # m: 0.01 .. 0.60
NEES_EDGES = np.array([0.05, 0.216, 0.5, 1.0, 2.0, 3.0, 5.0, 7.81, 9.35, 12.0, 20.0, 50.0])


# ---------------------------------------------------------------------------------------------- host emulation
def err2(traj, truth):
    """e^2 and e_xy^2 [rows][N] as the kernel forms them (no FMA), and whether the filter counts (finite)."""
    e = traj - truth
    exy = e[:, 0] * e[:, 0] + e[:, 1] * e[:, 1]
    e2 = exy + e[:, 2] * e[:, 2]
    return e2, exy, np.isfinite(e2)


def host_hist(val, ok, table):
    """[rows][len(table) + 1]: bin = number of table entries <= value, over the counted filters."""
    out = np.zeros((val.shape[0], len(table) + 1), dtype=np.uint64)
    for r in range(val.shape[0]):
        k = np.searchsorted(table, val[r][ok[r]], side="right")
        out[r] = np.bincount(k, minlength=len(table) + 1)
    return out


def nees_np(e, P, nd):
    """NEES of every filter: e [N][3], P [N][n][n]; (value, counted) with counted = positive LDL^T pivots."""
    S = P[:, :nd, :nd]
    ee = e[:, :nd]
    d0 = S[:, 0, 0]
    d1 = S[:, 1, 1] - S[:, 1, 0] / d0 * S[:, 1, 0]
    ok = (d0 > 0) & (d1 > 0) & np.isfinite(d0) & np.isfinite(d1)
    if nd == 3:
        l20 = S[:, 2, 0] / d0
        c = S[:, 2, 1] - l20 * S[:, 1, 0]
        d2 = S[:, 2, 2] - l20 * S[:, 2, 0] - c / d1 * c
        ok &= (d2 > 0) & np.isfinite(d2)
    val = np.zeros(len(e))
    if ok.any():
        val[ok] = np.einsum("ni,ni->n", ee[ok], np.linalg.solve(S[ok], ee[ok][..., None])[..., 0])
    ok &= np.isfinite(val) & np.isfinite(ee).all(axis=1)
    return np.where(ok, val, 0.0), ok


def step_reference(model, x0, r, anc, cfg, nd, truth_rows, K8=False):
    """Per-epoch NEES [rows][N] and whether it counts, from the covariance after each epoch (replayed epoch by
    epoch, the state read back in between)."""
    from roskfpos_b200.batch import Batch
    N = x0.shape[-1]
    nees, cnt = [], []
    with Batch(model, N, anchors=anc, **cfg) as b:
        b.set_state(x0)
        for t in range(r.shape[0]):
            if t:
                b.set_state(x, P)
            b.replay_toa(0.1, r[t:t + 1], err=0.01)
            x, P, _ = b.get_state()
            Pf = P.reshape(b.n, b.n, N).transpose(2, 0, 1)
            pz = np.full(N, 1.049) if K8 else x[2]
            v, ok = nees_np(np.stack([x[0], x[1], pz], axis=1) - truth_rows[t].T, Pf, nd)
            nees.append(v)
            cnt.append(ok)
    return np.array(nees), np.array(cnt)


def check_nees(got, nees, cnt, edges=NEES_EDGES):
    """Counts against the host binning of the numpy NEES (which matches the kernel's to ~1e-12): exact for every
    filter farther than 1e-9 relative from an edge; one near an edge may land on either side of it."""
    near = np.zeros_like(cnt)
    for e in edges:
        near |= np.abs(nees - e) <= 1e-9 * abs(e)
    near &= cnt
    ref = host_hist(nees, cnt & ~near, edges)
    diff = got.astype(np.int64) - ref.astype(np.int64)
    assert (diff >= 0).all()
    assert np.array_equal(diff.sum(axis=1), near.sum(axis=1))
    for r in np.nonzero(near.any(axis=1))[0]:
        allowed = set()
        for v in nees[r][near[r]]:
            j = int(np.argmin(np.abs(edges - v)))
            allowed |= {j, j + 1}
        assert set(np.nonzero(diff[r])[0]) <= allowed


def t6_case(N, T=6, m=8, seed=11, **rkw):
    anc = synth.anchors_for(m)
    truth = synth.truth_lissajous(N, T, 0.1, seed=seed)
    r = synth.ranges_mm(truth[1:], anc, seed=seed + 1, **rkw)
    return anc, truth, r


def run_hist(model, x0, r, anc, rows, cfg, quantities=("err", "err_xy", "nees"), edges=None):
    """One replay per quantity with the trajectory and that histogram registered: {quantity: counts}, plus the
    epoch_stats and traj of the last run."""
    from roskfpos_b200.batch import Batch
    N = x0.shape[-1]
    out = {}
    with Batch(model, N, anchors=anc, **cfg) as b:
        b.set_truth_traj(rows)
        for q in quantities:
            b.set_error_hist(edges if edges is not None else (NEES_EDGES if q == "nees" else EDGES), q)
            b.set_state(x0)
            out["traj"] = b.replay_toa(0.1, r, err=0.01, want_traj=True)[0]
            out[q] = b.error_hist()
            out["es"] = b.epoch_stats()
    return out


T6_CASES = [  # (m, wire format, config, range options)
    (8, np.int32, {}, {}),
    (8, np.uint16, {}, {}),
    (8, np.float64, {}, {}),
    (4, np.int32, {}, {}),
    (16, np.int32, {}, dict(p_missing=0.2)),
    (8, np.int32, dict(ignore_worst_anchor=1, ignore_cost_threshold=0.0), dict(p_nlos=0.2)),
    (8, np.int32, dict(variant=1, num_ignored_rangings=2), dict(p_nlos=0.2)),
    (8, np.int32, dict(variant=2), dict(p_nlos=0.2)),
]


@pytest.mark.parametrize("N", [4096, 1000, 129])
@pytest.mark.parametrize("case", range(len(T6_CASES)))
def test_t6_error_counts_exact(kflib, N, case):
    """ERR and ERR_XY counts equal np.searchsorted(edges**2, e2, "right") of traj against the truth exactly, and
    every row's total is epoch_stats column [2]; the NEES totals are column [5].  All wire formats, 4 / 8 / 16
    anchors, missing rangings, leave-one-out and the NLOS variants; N = 129 and 1000 leave partial warps."""
    m, dtype, cfg, rkw = T6_CASES[case]
    anc, truth, r = t6_case(N, m=m, **rkw)
    cfg = dict(accel_noise=0.5, **cfg)
    rr = r / 1000.0 if dtype == np.float64 else r.astype(dtype)
    got = run_hist(kflib.MODEL_T6, truth[0], rr, anc, truth[1:], cfg)
    e2, exy, fin = err2(got["traj"], truth[1:])
    assert np.array_equal(got["err"], host_hist(e2, fin, EDGES * EDGES))
    assert np.array_equal(got["err_xy"], host_hist(exy, fin, EDGES * EDGES))
    assert np.array_equal(got["err"].sum(axis=1), got["es"][:, 2].astype(np.uint64))
    assert np.array_equal(got["err_xy"].sum(axis=1), got["es"][:, 2].astype(np.uint64))
    assert np.array_equal(got["nees"].sum(axis=1), got["es"][:, 5].astype(np.uint64))
    assert (got["err"][:, 1:-1].sum(axis=1) > 0).all()  # the edges do spread the errors


@pytest.mark.parametrize("N", [4096, 1000, 129])
def test_t6_nees_counts(kflib, N):
    """NEES counts equal the host binning of the numpy NEES of the step-by-step reference (filters within 1e-9
    relative of an edge excepted); the totals equal epoch_stats column [5] exactly."""
    anc, truth, r = t6_case(N)
    cfg = dict(accel_noise=0.5)
    got = run_hist(kflib.MODEL_T6, truth[0], r, anc, truth[1:], cfg, quantities=("nees",))
    nees, cnt = step_reference(kflib.MODEL_T6, truth[0], r, anc, cfg, 3, truth[1:])
    assert np.array_equal(got["nees"].sum(axis=1), cnt.sum(axis=1).astype(np.uint64))
    assert np.array_equal(got["nees"].sum(axis=1), got["es"][:, 5].astype(np.uint64))
    check_nees(got["nees"], nees, cnt)


@pytest.mark.parametrize("model", ["K8", "T9"])
@pytest.mark.parametrize("N", [4096, 1000, 129])
def test_event_kernels(kflib, model, N):
    """K8 (z = the tag height, x-y NEES) and T9 through TOA schedules: ERR / ERR_XY exact, NEES against numpy,
    every total against epoch_stats."""
    anc, truth, r = t6_case(N)
    if model == "K8":
        mdl, nd, K8 = kflib.MODEL_K8, 2, True
        cfg = dict(xml=synth.K8_XML, accel_noise=0.5, jolt=0.5)
        x0 = np.zeros((8, N)); x0[:2] = truth[0][:2]
        rows = truth[1:].copy(); rows[:, 2] = 1.049
    else:
        mdl, nd, K8 = kflib.MODEL_T9, 3, False
        cfg = dict(accel_noise=0.5, jolt=0.5)
        x0 = np.zeros((9, N)); x0[:3] = truth[0]
        rows = truth[1:]
    got = run_hist(mdl, x0, r, anc, rows, cfg)
    tr = got["traj"].copy()
    if K8:
        tr[:, 2] = 1.049  # traj row 2 is the heading; the statistics use the tag height
    e2, exy, fin = err2(tr, rows)
    assert np.array_equal(got["err"], host_hist(e2, fin, EDGES * EDGES))
    assert np.array_equal(got["err_xy"], host_hist(exy, fin, EDGES * EDGES))
    assert np.array_equal(got["err"].sum(axis=1), got["es"][:, 2].astype(np.uint64))
    assert np.array_equal(got["nees"].sum(axis=1), got["es"][:, 5].astype(np.uint64))
    nees, cnt = step_reference(mdl, x0, r, anc, cfg, nd, rows, K8=K8)
    check_nees(got["nees"], nees, cnt)


def test_k8_multi_sensor_stream(kflib):
    """The full K8 event stream (IMU, PX4Flow, compass, TOA): one histogram row per TOA event, ERR counts exact
    against traj, totals against epoch_stats [2] and [5]."""
    from roskfpos_b200.batch import Batch
    N = 1000
    anc = synth.anchors_for(8)
    w = synth.k8_montecarlo_chunk(N, 0, 4, anc, "cuda:0", want_x0=True, want_truth_toa=True)
    rows = w["truth_toa"]
    res = {}
    with Batch(kflib.MODEL_K8, N, anchors=anc, xml=synth.K8_XML, accel_noise=0.5, jolt=0.5) as b:
        b.set_truth_traj(rows)
        for q in ("err", "nees"):
            b.set_error_hist(NEES_EDGES if q == "nees" else EDGES, q)
            b.set_state(w["x0"])
            traj = b.replay_events(w["events"], ranges=w["ranges"], sensors=w["sensors"], err=0.01, want_traj=True)
            res[q] = b.error_hist()
            es = b.epoch_stats()
    tr = traj.copy(); tr[:, 2] = 1.049
    e2, _, fin = err2(tr, rows.cpu().numpy())
    assert res["err"].shape == (w["n_toa"], len(EDGES) + 1)
    assert np.array_equal(res["err"], host_hist(e2, fin, EDGES * EDGES))
    assert np.array_equal(res["err"].sum(axis=1), es[:, 2].astype(np.uint64))
    assert np.array_equal(res["nees"].sum(axis=1), es[:, 5].astype(np.uint64))


@pytest.mark.parametrize("model", ["T6", "K8", "T9"])
def test_ragged_epochs_add_nothing(kflib, model):
    """replay_epochs (and, K8 / T9, replay_events_ragged): a filter whose dt < 0 in a row adds nothing there."""
    from roskfpos_b200.batch import Batch
    N, T = 1000, 6
    anc, truth, r = t6_case(N, T=T)
    rng = np.random.default_rng(3)
    dt = np.full((T, N), 0.1)
    skip = rng.random((T, N)) < 0.3
    dt[skip] = -1.0
    mdl = dict(T6=kflib.MODEL_T6, K8=kflib.MODEL_K8, T9=kflib.MODEL_T9)[model]
    cfg = dict(accel_noise=0.5) if model == "T6" else dict(accel_noise=0.5, jolt=0.5)
    if model == "K8":
        cfg["xml"] = synth.K8_XML
    n = dict(T6=6, K8=8, T9=9)[model]
    x0 = np.zeros((n, N)); x0[:3] = truth[0]
    rows = truth[1:].copy()
    if model == "K8":
        x0[2] = 0.0; rows[:, 2] = 1.049
    runs = []
    with Batch(mdl, N, anchors=anc, **cfg) as b:
        b.set_truth_traj(rows)
        b.set_error_hist(EDGES, "err")
        b.set_state(x0)
        runs.append((b.replay_epochs(dt, r, err=0.01, want_traj=True), b.error_hist(), b.epoch_stats()))
        if model != "T6":
            events = [(kflib.EV_TOA, 0.0, t * 8) for t in range(T)]
            b.set_state(x0)
            traj = b.replay_events(events, ranges=r.reshape(-1, N), err=0.01, want_traj=True, dt_per_filter=dt)
            runs.append((traj, b.error_hist(), b.epoch_stats()))
    for traj, h, es in runs:
        tr = traj.copy()
        if model == "K8":
            tr[:, 2] = 1.049
        e2, _, fin = err2(tr, rows)
        assert np.array_equal(h, host_hist(e2, fin & ~skip, EDGES * EDGES))
        assert np.array_equal(h.sum(axis=1), (~skip).sum(axis=1).astype(np.uint64))
        assert np.array_equal(h.sum(axis=1), es[:, 2].astype(np.uint64))


def test_non_interference(kflib):
    """epoch_stats, traj, sel, state, covariance, status and counters are bit-identical with and without a
    registered histogram (T6 leave-one-out, the K8 multi-sensor stream)."""
    from roskfpos_b200.batch import Batch
    N = 1000
    anc, truth, r = t6_case(N, p_nlos=0.2)
    outs = []
    for on in (False, True):
        with Batch(kflib.MODEL_T6, N, anchors=anc, accel_noise=0.5, ignore_worst_anchor=1) as b:
            b.set_truth_traj(truth[1:])
            if on:
                b.set_error_hist(EDGES, "err")
            b.set_truth(truth[-1])
            b.set_state(truth[0])
            traj, sel = b.replay_toa(0.1, r, err=0.01, want_traj=True, want_sel=True)
            x, P, st = b.get_state()
            outs.append(dict(traj=traj, sel=sel, x=x, P=P, st=st, cnt=b.counters(), fin=b.error_stats(),
                             es=b.epoch_stats()))
    a, c = outs
    for k in ("traj", "sel", "x", "P", "st", "fin", "es"):
        assert np.array_equal(a[k], c[k]), k
    assert a["cnt"] == c["cnt"]
    w = synth.k8_workload(N, 3, anc, seed=5, full=True)
    base = None
    for on in (False, True):
        with Batch(kflib.MODEL_K8, N, anchors=anc, xml=synth.K8_XML, accel_noise=0.5, jolt=0.5) as b:
            b.set_truth_traj(np.repeat(w["truth_end"][None], w["n_toa"], axis=0))
            if on:
                b.set_error_hist(NEES_EDGES, "nees")
            b.set_state(w["x0"])
            traj = b.replay_events(w["events"], ranges=w["ranges"], sensors=w["sensors"], err=0.01, want_traj=True)
            x, P, st = b.get_state()
            res = (traj, x, P, st, b.epoch_stats(), b.counters())
        if base is not None:
            for u, v in zip(res[:5], base[:5]):
                assert np.array_equal(u, v)
            assert res[5] == base[5]
        base = res


def test_chunking_and_reruns(kflib):
    """One replay of T rows gives the counts of two replays of T/2; a re-run after set_state overwrites the rows
    (it does not add to them); rows the cursor has not reached read zero; the histogram survives a truth
    re-registration, which zeroes it."""
    from roskfpos_b200.batch import Batch
    N, T = 1000, 8
    anc, truth, r = t6_case(N, T=T)
    with Batch(kflib.MODEL_T6, N, anchors=anc, accel_noise=0.5) as b:
        b.set_error_hist(EDGES, "err")  # first the histogram, then the truth: both orders allocate
        b.set_truth_traj(truth[1:])
        b.set_state(truth[0])
        b.replay_toa(0.1, r, err=0.01)
        whole = b.error_hist()
        b.set_state(truth[0])
        b.replay_toa(0.1, r[:T // 2], err=0.01)
        half = b.error_hist()
        b.replay_toa(0.1, r[T // 2:], err=0.01)
        two = b.error_hist()
        b.set_state(truth[0])
        for t in range(T):
            b.step_toa(0.1, r[t], err=0.01)
        stepped = b.error_hist()
        dev = b.error_hist(readback=False)
        b.set_truth_traj(truth[1:])
        fresh = b.error_hist()
    assert whole.sum() == N * T
    assert np.array_equal(whole, two) and np.array_equal(whole, stepped)
    assert np.array_equal(dev.cpu().numpy().astype(np.uint64), whole)
    assert np.array_equal(half[:T // 2], whole[:T // 2]) and (half[T // 2:] == 0).all()
    assert (fresh == 0).all() and fresh.shape == whole.shape


def test_sharding_and_allreduce(kflib):
    """toa_montecarlo shards with arbitrary first_filter splits sum to the whole batch's counts exactly (chunked
    or not); error_hist_allreduce alone and through a one-rank NCCL communicator equals error_hist."""
    from roskfpos_b200.batch import Batch
    from roskfpos_b200.shard import nccl_comm
    N, T = 4099, 12
    anc = synth.anchors_for(8)
    kw = dict(p_missing=0.05, p_nlos=0.05)

    def run(lo, hi, chunk, q="err"):
        with Batch(kflib.MODEL_T6, hi - lo, anchors=anc, accel_noise=0.5) as b:
            return synth.toa_montecarlo(b, T, chunk, anc, first_filter=lo,
                                        hist=(NEES_EDGES if q == "nees" else EDGES, q), **kw)
    rows, whole = run(0, N, T)
    assert whole.shape == (T, len(EDGES) + 1) and np.array_equal(whole.sum(axis=1), rows[:, 2].astype(np.uint64))
    assert np.array_equal(run(0, N, 5)[1], whole)
    cuts = [0, 1000, 3001, 3002, N]
    parts = [run(lo, hi, 7)[1] for lo, hi in zip(cuts[:-1], cuts[1:])]
    assert np.array_equal(sum(p.astype(np.uint64) for p in parts), whole)
    nw = run(0, N, T, "nees")[1]
    assert np.array_equal(sum(run(lo, hi, T, "nees")[1] for lo, hi in ((0, 1234), (1234, N))), nw)
    anc_t, truth, r = t6_case(2048, seed=21)
    comm = nccl_comm(0, 1, 0)
    try:
        with Batch(kflib.MODEL_T6, 2048, anchors=anc_t, accel_noise=0.5) as b:
            b.set_truth_traj(truth[1:]); b.set_error_hist(EDGES, "err_xy")
            b.set_state(truth[0]); b.replay_toa(0.1, r, err=0.01)
            ref = b.error_hist()
            red = b.error_hist_allreduce(comm)
            alone = b.error_hist_allreduce(None)
    finally:
        comm.close()
    assert np.array_equal(red, ref) and np.array_equal(alone, ref) and ref.sum() == 2048 * r.shape[0]


WORKER = textwrap.dedent("""
    import sys
    import numpy as np
    sys.path.insert(0, %r)
    import torch
    import torch.distributed as dist
    from roskfpos_b200 import lib as L, synth
    from roskfpos_b200.batch import Batch
    from roskfpos_b200.shard import nccl_comm
    dist.init_process_group("gloo")
    rank, world = dist.get_rank(), dist.get_world_size()
    torch.cuda.set_device(rank)
    N, T, cut = 3001, 6, 1234
    anc = synth.anchors_for(8)
    edges = np.arange(1, 61) * 0.01
    lo, hi = (0, cut) if rank == 0 else (cut, N)
    w = synth.toa_montecarlo_chunk(hi - lo, 0, T, anc, "cuda:%%d" %% rank, first_filter=lo, want_x0=True,
                                   want_truth=True)
    comm = nccl_comm(rank, world, rank)
    with Batch(L.MODEL_T6, hi - lo, device=rank, anchors=anc, accel_noise=0.5) as b:
        b.set_truth_traj(w["truth"]); b.set_error_hist(edges, "err")
        b.set_state(w["x0"]); b.replay_toa(w["dt"], w["ranges"], err=0.01)
        red = b.error_hist_allreduce(comm)
    comm.close()
    if rank == 0:
        with Batch(L.MODEL_T6, N, device=0, anchors=anc, accel_noise=0.5) as b:
            _, whole = synth.toa_montecarlo(b, T, T, anc, hist=(edges, "err"))
        print("RESULT", int(np.array_equal(red, whole)), int(red.sum()))
    dist.destroy_process_group()
""")


def test_allreduce_two_ranks(kflib, tmp_path):
    """Two ranks on two GPUs with unequal shards: the NCCL allreduce equals the single-batch counts."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    script = tmp_path / "worker.py"
    script.write_text(WORKER % ROOT)
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
           "--master-addr", "127.0.0.1", "--master-port", str(port), str(script)]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = [l for l in out.stdout.splitlines() if l.startswith("RESULT")][-1]
    assert line.split()[1:] == ["1", str(3001 * 6)]


def test_errors(kflib):
    """ML batch, bad quantity, non-increasing / non-finite / negative-metre edges, 256 edges: INVALID; 0 edges
    unregisters; reading with nothing (or only one of histogram and truth) registered: NOT_READY; a row count
    that differs from the registration: INVALID."""
    from roskfpos_b200.batch import Batch
    N = 256
    anc, truth, r = t6_case(N)
    lib = kflib.lib()

    def reg(b, q, e):
        e = np.ascontiguousarray(e, dtype=np.float64)
        return lib.kfpos_batch_set_error_hist(b._h, q, len(e), C.c_void_p(e.ctypes.data))
    out = np.zeros((6, len(EDGES) + 1), dtype=np.uint64)

    def read(b, rows=6):
        return lib.kfpos_batch_error_hist(b._h, rows, C.c_void_p(out.ctypes.data), None)
    with Batch(kflib.MODEL_ML, N, anchors=anc) as b:
        assert reg(b, kflib.HIST_ERR, EDGES) == INVALID
    with Batch(kflib.MODEL_T6, N, anchors=anc, accel_noise=0.5) as b:
        assert read(b) == NOT_READY
        for q in (-1, 3):
            assert reg(b, q, EDGES) == INVALID
        assert reg(b, kflib.HIST_ERR, [0.1, 0.1, 0.2]) == INVALID
        assert reg(b, kflib.HIST_ERR, [0.2, 0.1]) == INVALID
        assert reg(b, kflib.HIST_ERR, [0.1, np.nan]) == INVALID
        assert reg(b, kflib.HIST_NEES, [0.1, np.inf]) == INVALID
        assert reg(b, kflib.HIST_ERR_XY, [-0.1, 0.1]) == INVALID
        assert reg(b, kflib.HIST_ERR, np.arange(1, 257) * 0.01) == INVALID
        assert reg(b, kflib.HIST_NEES, np.arange(-5, 250) * 0.5) == 0  # 255 edges, NEES may start below 0
        assert reg(b, kflib.HIST_ERR, np.arange(1, 256) * 0.01) == 0
        assert reg(b, kflib.HIST_ERR, EDGES) == 0
        assert read(b) == NOT_READY  # no truth trajectory yet
        b.set_truth_traj(truth[1:])
        assert read(b) == 0 and (out == 0).all()
        assert read(b, 5) == INVALID
        e = np.ascontiguousarray(EDGES)
        assert lib.kfpos_batch_set_error_hist(b._h, kflib.HIST_ERR, 0, C.c_void_p(e.ctypes.data)) == 0
        assert read(b) == NOT_READY  # 0 edges unregistered it
        assert reg(b, kflib.HIST_ERR, EDGES) == 0
        b.set_truth_traj(None)
        assert read(b) == NOT_READY
        b.set_state(truth[0])
        b.replay_toa(0.1, r, err=0.01)  # a histogram without a trajectory runs the plain kernel
        b.set_error_hist(None)
        with pytest.raises(ValueError):
            b.set_error_hist(EDGES, "rmse")
