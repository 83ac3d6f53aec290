"""GPU: per-epoch Monte Carlo statistics (kfpos_batch_set_truth_traj / kfpos_batch_epoch_stats) fused into the
T6, K8 and T9 replay kernels -- the documented summation tree reproduced on the host bit for bit, NEES against
numpy, RMSE(t) against the CPU oracle, ragged epochs, non-interference with everything else a replay produces,
chunking, sharding, the device truth generator and the error paths."""
import numpy as np
import pytest

from roskfpos_b200 import synth

pytestmark = pytest.mark.gpu

INVALID, NOT_READY = -1, -4


# ---------------------------------------------------------------------------------------------- host emulation
def terms(traj, truth, skip=None):
    """Columns 0..2 of every filter and row: [rows][N][3] (no FMA: numpy evaluates what the kernel does)."""
    e = traj - truth
    exy = e[:, 0] * e[:, 0] + e[:, 1] * e[:, 1]
    e2 = exy + e[:, 2] * e[:, 2]
    fin = np.isfinite(e2)
    v = np.stack([np.where(fin, e2, 0.0), np.where(fin, exy, 0.0), fin * 1.0], axis=-1)
    if skip is not None:
        v[skip] = 0.0
    return v


def tree(v):
    """The documented order: per 32-filter warp a 32-leaf tree (lane i += lane i + s, s = 16 .. 1, missing lanes
    = 0), then the pairwise tree over the warp index.  v [rows][N][W] -> [rows][W]."""
    rows, N, W = v.shape
    nw = (N + 31) // 32
    a = np.zeros((rows, nw * 32, W))
    a[:, :N] = v
    a = a.reshape(rows, nw, 32, W)
    for s in (16, 8, 4, 2, 1):
        a[:, :, :s] = a[:, :, :s] + a[:, :, s:2 * s]
    w = a[:, :, 0].copy()
    stride = 1
    while stride < nw:
        i = np.arange(0, nw - stride, 2 * stride)
        w[:, i] = w[:, i] + w[:, i + stride]
        stride *= 2
    return w[:, 0]


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


def t6_case(N, T=6, m=8, seed=11, **rkw):
    anc = synth.anchors_for(m)
    truth = synth.truth_lissajous(N, T, 0.1, seed=seed)
    r = synth.ranges_mm(truth[1:], anc, seed=seed + 1, **rkw)
    return anc, truth, r


def step_reference(kflib, model, x0, r, anc, cfg, nd, truth_rows, K8=False):
    """Replays epoch by epoch, restoring (x, P) before each one so that the status word is that epoch's:
    per row (status != 0, NEES terms) from the covariance the filter holds after the epoch."""
    from roskfpos_b200.batch import Batch
    N = x0.shape[-1]
    bad, nees, cnt = [], [], []
    with Batch(model, N, anchors=anc, **cfg) as b:
        b.set_state(x0)
        for t in range(r.shape[0]):
            if t:
                b.set_state(x, P)
            b.replay_toa(0.1, r[t:t + 1], err=0.01)
            x, P, st = b.get_state()
            n = b.n
            Pf = P.reshape(n, n, N).transpose(2, 0, 1)
            pz = np.full(N, 1.049) if K8 else x[2]
            e = np.stack([x[0], x[1], pz], axis=1) - truth_rows[t].T
            v, ok = nees_np(e, Pf, nd)
            bad.append(st != 0)
            nees.append(v)
            cnt.append(ok * 1.0)
    return np.array(bad), np.array(nees), np.array(cnt)


def run_es(kflib, model, x0, r, anc, truth_rows, cfg):
    """One replay with the trajectory registered: dict(es = epoch_stats, traj, sel, state, counters)."""
    from roskfpos_b200.batch import Batch
    N = x0.shape[-1]
    with Batch(model, N, anchors=anc, **cfg) as b:
        b.set_truth_traj(truth_rows)
        b.set_state(x0)
        traj, sel = b.replay_toa(0.1, r, err=0.01, want_traj=True, want_sel=model == kflib.MODEL_T6)
        es = b.epoch_stats()
        x, P, st = b.get_state()
        cnt = b.counters()
    return dict(es=es, traj=traj, sel=sel, x=x, P=P, st=st, cnt=cnt)


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
def test_t6_exact_sums_and_nees(kflib, N, case):
    """Columns 0..3 equal the host emulation of the documented tree bit for bit; column 4 the numpy NEES to
    1e-12 relative, column 5 exactly.  All wire formats, 4 / 8 / 16 anchors, missing rangings, leave-one-out and
    the NLOS variants; N = 129 and 1000 leave partial warps."""
    m, dtype, cfg, rkw = T6_CASES[case]
    anc, truth, r = t6_case(N, m=m, **rkw)
    cfg = dict(accel_noise=0.5, **cfg)
    rr = r / 1000.0 if dtype == np.float64 else r.astype(dtype)  # the wire format of the case
    got = run_es(kflib, kflib.MODEL_T6, truth[0], rr, anc, truth[1:], cfg)
    bad, nees, cnt = step_reference(kflib, kflib.MODEL_T6, truth[0], rr, anc, cfg, 3, truth[1:])
    v = terms(got["traj"], truth[1:])
    ref = tree(np.concatenate([v, bad[..., None] * 1.0], axis=-1))
    assert np.array_equal(got["es"][:, :4], ref)
    ref_n = tree(np.stack([nees, cnt], axis=-1))
    assert np.array_equal(got["es"][:, 5], ref_n[:, 1])
    assert np.allclose(got["es"][:, 4], ref_n[:, 0], rtol=1e-12, atol=0)
    assert (got["es"][:, 2] == N).all() and (got["es"][:, 5] > 0).all()


@pytest.mark.parametrize("model", ["K8", "T9"])
@pytest.mark.parametrize("N", [4096, 1000, 129])
def test_event_kernels_exact_sums_and_nees(kflib, model, N):
    """K8 (x-y NEES, z = tag height) and T9 through TOA schedules: columns 0..3 bit for bit, NEES to 1e-12."""
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
    got = run_es(kflib, mdl, x0, r, anc, rows, cfg)
    bad, nees, cnt = step_reference(kflib, mdl, x0, r, anc, cfg, nd, rows, K8=K8)
    tr = got["traj"].copy()
    if K8:
        tr[:, 2] = 1.049  # traj row 2 is the heading; the statistics use the tag height
    v = terms(tr, rows)
    assert np.array_equal(got["es"][:, :4], tree(np.concatenate([v, bad[..., None] * 1.0], axis=-1)))
    ref_n = tree(np.stack([nees, cnt], axis=-1))
    assert np.array_equal(got["es"][:, 5], ref_n[:, 1])
    assert np.allclose(got["es"][:, 4], ref_n[:, 0], rtol=1e-12, atol=0)


def test_k8_multi_sensor_schedule(kflib):
    """The full K8 event stream (IMU, PX4Flow, compass, TOA): one row per TOA event, columns 0..2 bit for bit
    against the emulation on `traj`; the last row agrees with the final-state error_stats."""
    from roskfpos_b200.batch import Batch
    N = 1000
    anc = synth.anchors_for(8)
    w = synth.k8_montecarlo_chunk(N, 0, 4, anc, "cuda:0", want_x0=True, want_truth_toa=True)
    rows = w["truth_toa"]
    with Batch(kflib.MODEL_K8, N, anchors=anc, xml=synth.K8_XML, accel_noise=0.5, jolt=0.5) as b:
        b.set_truth_traj(rows)
        b.set_truth(w["truth_end"])
        b.set_state(w["x0"])
        traj = b.replay_events(w["events"], ranges=w["ranges"], sensors=w["sensors"], err=0.01, want_traj=True)
        es = b.epoch_stats()
        fin = b.error_stats()
    tr = traj.copy(); tr[:, 2] = 1.049
    v = terms(tr, rows.cpu().numpy())
    assert es.shape == (w["n_toa"], 6)
    assert np.array_equal(es[:, :3], tree(v))
    assert es[-1, 2] == fin[2] and abs(es[-1, 0] - fin[0]) <= 1e-13 * fin[0]
    assert (es[:, 3] <= N).all() and (es[:, 5] > 0).all()


def test_rmse_against_the_oracle(kflib, oracle):
    """RMSE(t) of the statistics agrees with RMSE(t) of the CPU oracle's trajectory (T6, K8, T9) to 1e-9."""
    from roskfpos_b200.batch import Batch, epoch_summary
    N = 2048
    anc, truth, r = t6_case(N, T=10)
    rows = truth[1:]

    def rmse(traj, rw):
        e = traj - rw
        return np.sqrt((e ** 2).sum(axis=1).mean(axis=1))
    with Batch(kflib.MODEL_T6, N, anchors=anc, accel_noise=0.5) as b:
        b.set_truth_traj(rows); b.set_state(truth[0]); b.replay_toa(0.1, r, err=0.01)
        got = epoch_summary(b.epoch_stats())["rmse"]
    ref = oracle.t6_replay(truth[0], None, r, anc, 0.1, 0.01, want_traj=True)["traj"]
    assert np.allclose(got, rmse(ref, rows), rtol=1e-9, atol=0)
    x9 = np.zeros((9, N)); x9[:3] = truth[0]
    events = [(0, 0.1, t * 8) for t in range(10)]
    with Batch(kflib.MODEL_T9, N, anchors=anc, accel_noise=0.5, jolt=0.5) as b:
        b.set_truth_traj(rows); b.set_state(x9)
        b.replay_events(events, ranges=r.reshape(-1, N), err=0.01)
        got = epoch_summary(b.epoch_stats())["rmse"]
    ref = oracle.t9_events(x9, None, events, r.reshape(-1, N), None, anc, 0.01, want_traj=True)["traj"]
    assert np.allclose(got, rmse(ref, rows), rtol=1e-9, atol=0)
    w = synth.k8_workload(N, 4, anc, seed=5, full=True)
    with Batch(kflib.MODEL_K8, N, anchors=anc, xml=synth.K8_XML, accel_noise=0.5, jolt=0.5) as b:
        b.set_state(w["x0"])
        traj = b.replay_events(w["events"], ranges=w["ranges"], sensors=w["sensors"], err=0.01, want_traj=True)
    kref = oracle.k8_replay(w["x0"], None, w["events"], w["ranges"], w["sensors"], anc, 0.01,
                            oracle.k8_cfg(0.5, 0.5, **synth.K8_ORACLE_CFG), want_traj=True)["traj"]
    # the K8 truth rows are not needed to compare the two trajectories' errors: use the GPU's own as truth
    krows = traj.copy(); krows[:, 2] = 1.049
    with Batch(kflib.MODEL_K8, N, anchors=anc, xml=synth.K8_XML, accel_noise=0.5, jolt=0.5) as b:
        b.set_truth_traj(krows + 0.25); b.set_state(w["x0"])
        b.replay_events(w["events"], ranges=w["ranges"], sensors=w["sensors"], err=0.01)
        got = epoch_summary(b.epoch_stats())["rmse"]
    kr = kref.copy(); kr[:, 2] = 1.049
    assert np.allclose(got, rmse(kr, krows + 0.25), rtol=1e-9, atol=0)


@pytest.mark.parametrize("model", ["T6", "K8", "T9"])
def test_ragged_epochs_add_nothing(kflib, model):
    """replay_epochs / replay_events_ragged: a filter whose dt < 0 in a row adds nothing to that row."""
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
    with Batch(mdl, N, anchors=anc, **cfg) as b:
        b.set_truth_traj(rows)
        b.set_state(x0)
        traj = b.replay_epochs(dt, r, err=0.01, want_traj=True)
        es = b.epoch_stats()
    tr = traj.copy()
    if model == "K8":
        tr[:, 2] = 1.049
    v = terms(tr, rows, skip=skip)
    assert np.array_equal(es[:, :3], tree(v))
    assert np.array_equal(es[:, 2], (~skip).sum(axis=1) * 1.0)
    assert (es[:, 5] <= es[:, 2]).all()


def test_non_interference(kflib):
    """State, covariance, status, traj, sel, counters and the final-state error_stats are bit-identical with the
    statistics on and off; the last row's n equals error_stats n and its sum |e|^2 agrees to 1e-13."""
    from roskfpos_b200.batch import Batch
    N = 1000
    anc, truth, r = t6_case(N, p_nlos=0.2)
    outs = []
    for on in (False, True):
        with Batch(kflib.MODEL_T6, N, anchors=anc, accel_noise=0.5, ignore_worst_anchor=1) as b:
            if on:
                b.set_truth_traj(truth[1:])
            b.set_truth(truth[-1])
            b.set_state(truth[0])
            traj, sel = b.replay_toa(0.1, r, err=0.01, want_traj=True, want_sel=True)
            x, P, st = b.get_state()
            outs.append(dict(traj=traj, sel=sel, x=x, P=P, st=st, cnt=b.counters(), fin=b.error_stats(),
                             es=b.epoch_stats() if on else None))
    a, c = outs
    for k in ("traj", "sel", "x", "P", "st", "fin"):
        assert np.array_equal(a[k], c[k]), k
    assert a["cnt"] == c["cnt"]
    assert c["es"][-1, 2] == c["fin"][2]
    assert abs(c["es"][-1, 0] - c["fin"][0]) <= 1e-13 * c["fin"][0]
    # K8 / T9
    w = synth.k8_workload(N, 3, anc, seed=5, full=True)
    for on in (False, True):
        with Batch(kflib.MODEL_K8, N, anchors=anc, xml=synth.K8_XML, accel_noise=0.5, jolt=0.5) as b:
            if on:
                b.set_truth_traj(np.repeat(w["truth_end"][None], w["n_toa"], axis=0))
            b.set_truth(w["truth_end"])
            b.set_state(w["x0"])
            traj = b.replay_events(w["events"], ranges=w["ranges"], sensors=w["sensors"], err=0.01, want_traj=True)
            x, P, st = b.get_state()
            res = (traj, x, P, st, b.counters(), b.error_stats())
        if on:
            for u, v in zip(res[:4], base[:4]):
                assert np.array_equal(u, v)
            assert res[4] == base[4] and np.array_equal(res[5], base[5])
        base = res


def test_chunking_and_cursor(kflib):
    """One replay of T rows equals two replays of T/2 under one registration bit for bit; set_state resets the
    cursor (rows not reached read zero); a launch past the registered rows is refused and runs nothing."""
    from roskfpos_b200.batch import Batch
    N, T = 1000, 8
    anc, truth, r = t6_case(N, T=T)
    with Batch(kflib.MODEL_T6, N, anchors=anc, accel_noise=0.5) as b:
        b.set_truth_traj(truth[1:])
        b.set_state(truth[0])
        b.replay_toa(0.1, r, err=0.01)
        whole = b.epoch_stats()
        b.set_state(truth[0])
        b.replay_toa(0.1, r[:T // 2], err=0.01)
        half = b.epoch_stats()
        b.replay_toa(0.1, r[T // 2:], err=0.01)
        two = b.epoch_stats()
        x_before, _, _ = b.get_state()
        with pytest.raises(kflib.KfposError) as ei:
            b.step_toa(0.1, r[0], err=0.01)
        assert ei.value.code == INVALID
        x_after, _, _ = b.get_state()
        assert np.array_equal(x_before, x_after)
        # step_toa advances the cursor one row at a time
        b.set_state(truth[0])
        for t in range(T):
            b.step_toa(0.1, r[t], err=0.01)
        stepped = b.epoch_stats()
    assert np.array_equal(whole, two) and np.array_equal(whole, stepped)
    assert np.array_equal(half[:T // 2], whole[:T // 2]) and (half[T // 2:] == 0).all()


def test_sharding_and_allreduce(kflib):
    """Aligned shards of N / G filters folded pairwise in rank order equal the whole batch bit for bit; the
    allreduce through a one-rank NCCL communicator equals epoch_stats."""
    from roskfpos_b200.batch import Batch
    from roskfpos_b200.shard import nccl_comm
    N = 8192
    anc, truth, r = t6_case(N, seed=21)

    def stats(lo, hi):
        with Batch(kflib.MODEL_T6, hi - lo, anchors=anc, accel_noise=0.5) as b:
            b.set_truth_traj(np.ascontiguousarray(truth[1:, :, lo:hi]))
            b.set_state(np.ascontiguousarray(truth[0][:, lo:hi]))
            b.replay_toa(0.1, np.ascontiguousarray(r[:, :, lo:hi]), err=0.01)
            return b.epoch_stats()
    whole = stats(0, N)
    for G in (2, 4, 8):
        parts = [stats(g * N // G, (g + 1) * N // G) for g in range(G)]
        stride = 1
        while stride < G:
            for i in range(0, G - stride, 2 * stride):
                parts[i] = parts[i] + parts[i + stride]
            stride *= 2
        assert np.array_equal(parts[0], whole), G
    comm = nccl_comm(0, 1, 0)
    try:
        with Batch(kflib.MODEL_T6, N, anchors=anc, accel_noise=0.5) as b:
            b.set_truth_traj(truth[1:]); b.set_state(truth[0]); b.replay_toa(0.1, r, err=0.01)
            red = b.epoch_stats_allreduce(comm)
            alone = b.epoch_stats_allreduce(None)
    finally:
        comm.close()
    assert np.array_equal(red, whole) and np.array_equal(alone, whole)


def test_device_truth_generators(kflib):
    """kfpos_synth_k8_truth at the chunk's last TOA event (its end time) equals truth_end of kfpos_synth_k8 bit
    for bit, chunk by chunk; device_truth_traj's last row equals device_ranges_mm's truth_end."""
    anc = synth.anchors_for(8)
    for macro0 in (0, 3):
        w = synth.k8_montecarlo_chunk(777, macro0, 3, anc, "cuda:0", first_filter=5000, want_truth_toa=True)
        assert w["truth_toa"].shape == (w["n_toa"], 3, 777)
        assert (w["truth_toa"][-1] == w["truth_end"]).all().item()
    _, x0, tend = synth.device_ranges_mm(300, 5, anc, 0.1, "cuda:0", step0=7)
    tt = synth.device_truth_traj(300, 5, 0.1, "cuda:0", step0=7)
    assert (tt[-1] == tend).all().item()


def test_errors(kflib):
    """epoch_stats before any registration: NOT_READY; a row count that differs from the registration: INVALID;
    an ML batch: INVALID; unregistering stops the statistics."""
    from roskfpos_b200.batch import Batch
    import ctypes as C
    N = 256
    anc, truth, r = t6_case(N)
    out = np.zeros((6, 6))
    with Batch(kflib.MODEL_T6, N, anchors=anc, accel_noise=0.5) as b:
        rc = kflib.lib().kfpos_batch_epoch_stats(b._h, 6, C.c_void_p(out.ctypes.data), None)
        assert rc == NOT_READY
        b.set_truth_traj(truth[1:])
        assert kflib.lib().kfpos_batch_epoch_stats(b._h, 5, C.c_void_p(out.ctypes.data), None) == INVALID
        b.set_state(truth[0])
        with pytest.raises(kflib.KfposError) as ei:
            b.replay_toa(0.1, np.concatenate([r, r[:1]]), err=0.01)
        assert ei.value.code == INVALID
        assert (b.epoch_stats() == 0).all()
        b.set_truth_traj(None)
        b.replay_toa(0.1, np.concatenate([r, r[:1]]), err=0.01)
    with Batch(kflib.MODEL_ML, N, anchors=anc) as b:
        assert kflib.lib().kfpos_batch_set_truth_traj(b._h, 6, C.c_void_p(truth.ctypes.data), None) == INVALID
