"""Rangings along any trajectory (DESIGN §4.5g): kfpos_synth_toa_ranges_truth writes the log of the Lissajous
generator byte for byte when it is given the Lissajous truth, the random walk of kfpos_synth_walk equals a numpy
restatement of its step bit for bit and has the documented statistics, it is pure under sharding and chunking, and
the Monte Carlo bench runs on it."""
import ctypes as C

import numpy as np
import pytest

from roskfpos_b200 import lib as L, synth
from tests.test_gpu_synth_geo import STUDY, bits, geo_uniforms, slab, table
from tests.test_gpu_synth_toa import oracle_t6, t6_run
from tests.util import assert_parity, to_metres, ulp_perturbations

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
INF = float("inf")
# the room walk of the DESIGN §4.5g study: z held at the centre of (0.5, 1.5), 1.0 m
ROOM_WALK = dict(accel_sd=(0.5, 0.5, 0.0), v_max=(1.5, 1.5, INF), lo=(0.5, 0.5, 0.5), hi=(9.5, 9.5, 1.5))


def walk(n, epoch0, T, state=None, **kw):
    """synth.walk_truth_chunk with the room walk by default: host (truth, state, x0 or None)."""
    kw = dict(dict(seed=synth.SEED, period=0.1, **ROOM_WALK), **kw)
    w = synth.walk_truth_chunk(n, epoch0, T, DEV, state=state, **kw)
    x0 = w.get("x0")
    return w["truth"].cpu().numpy(), w["state"].cpu().numpy(), None if x0 is None else x0.cpu().numpy()


def truth_call(n, epoch0, truth, boxes=(), fmt=L.FMT_I32_MM, anc=None, seed=synth.SEED, first_filter=0, **kw):
    """kfpos_synth_toa_ranges_truth through the C ABI: `truth` a host array or a device tensor; host (ranges, nlos)."""
    import torch
    anc = np.ascontiguousarray(synth.anchors_for(8) if anc is None else anc, dtype=np.float64)
    T, M = truth.shape[0], len(anc)
    r = torch.empty((T, M, n), dtype=torch.uint16 if fmt == L.FMT_U16_MM else torch.int32, device=DEV)
    m = torch.empty((T, n), dtype=torch.int32, device=DEV)
    g = L.KfposSynthToa(**dict(dict(seed=seed, first_filter=first_filter, first_epoch=epoch0, tag_z=-7.0,
                                    sigma_r=0.1, nlos_mean=0.8), **kw))
    boxes = np.asarray(boxes, dtype=np.float64).reshape(-1, 9)
    tp = C.c_void_p(truth.data_ptr()) if isinstance(truth, torch.Tensor) else C.c_void_p(truth.ctypes.data)
    L.check(L.lib().kfpos_synth_toa_ranges_truth(0, n, M, C.c_void_p(anc.ctypes.data), T, tp, C.byref(g), len(boxes),
                                                 C.cast(table(boxes), C.c_void_p) if len(boxes) else None, fmt,
                                                 C.c_void_p(r.data_ptr()), C.c_void_p(m.data_ptr()), None),
            "kfpos_synth_toa_ranges_truth")
    return r.cpu().numpy(), m.cpu().numpy().view(np.uint32)


def np_walk(x, v, T, dt, lo, hi, v_max, acc=None):
    """numpy restatement of the step (single IEEE operations): positions [T][3][N] and the final (x, v)."""
    lo, hi, v_max = (np.asarray(a, dtype=np.float64)[:, None] for a in (lo, hi, v_max))
    h = dt * dt / 2.0
    out = []
    for k in range(T):
        a = np.zeros_like(x) if acc is None else acc[k]
        xn = (x + v * dt) + a * h
        vn = v + a * dt
        up = xn > hi
        dn = ~up & (xn < lo)
        xn = np.where(up, (hi + hi) - xn, np.where(dn, (lo + lo) - xn, xn))
        vn = np.where(up | dn, -vn, vn)
        x, v = np.fmin(np.fmax(xn, lo), hi), np.fmin(np.fmax(vn, -v_max), v_max)
        out.append(x)
    return np.stack(out), x, v


# ------------------------------------------------------------------------- 1. byte identity with the Lissajous
@pytest.mark.parametrize("fmt", [L.FMT_I32_MM, L.FMT_U16_MM])
@pytest.mark.parametrize("impair", [False, True])
def test_lissajous_truth_gives_the_same_bytes(fmt, impair):
    """The truth of kfpos_synth_k8_truth at the epoch times, handed to kfpos_synth_toa_ranges_truth, gives the log
    and mask of kfpos_synth_toa_ranges / _nlos / _geo: with 0 and 3 boxes, host and device truth, and a call of
    more than the 1024 epochs of one launch."""
    N, T, epoch0 = 3000, 1100, 7
    kw = dict(p_missing=0.05, p_nlos=0.05) if impair else {}
    anc = synth.anchors_for(8)
    ref = synth.toa_montecarlo_chunk(N, epoch0, T, anc, DEV, fmt=fmt, want_truth=True, want_nlos=True, **kw)
    truth = ref["truth"]
    r0, m0 = ref["ranges"].cpu().numpy(), ref["nlos"].cpu().numpy().view(np.uint32)
    plain = synth.toa_montecarlo_chunk(N, epoch0, T, anc, DEV, fmt=fmt, **kw)["ranges"].cpu().numpy()
    assert np.array_equal(plain, r0)
    for src in (truth, truth.cpu().numpy()):
        r, m = truth_call(N, epoch0, src, fmt=fmt, **kw)
        assert np.array_equal(r, r0) and np.array_equal(m, m0)
    g = synth.toa_montecarlo_chunk(N, epoch0, T, anc, DEV, fmt=fmt, want_nlos=True, obstacles=STUDY, **kw)
    rg, mg = g["ranges"].cpu().numpy(), g["nlos"].cpu().numpy().view(np.uint32)
    assert not np.array_equal(mg, m0)
    for src in (truth, truth.cpu().numpy()):
        r, m = truth_call(N, epoch0, src, boxes=STUDY, fmt=fmt, **kw)
        assert np.array_equal(r, rg) and np.array_equal(m, mg)
    # the Python path, with the truth tensor handed back
    w = synth.toa_montecarlo_chunk(N, epoch0, T, anc, DEV, fmt=fmt, want_nlos=True, want_truth=True, obstacles=STUDY,
                                   truth=truth, tag_z=123.0, **kw)
    assert np.array_equal(w["ranges"].cpu().numpy(), rg) and np.array_equal(w["nlos"].cpu().numpy().view(np.uint32), mg)
    assert w["truth"] is truth
    assert np.array_equal(w["truth_end"].cpu().numpy(), truth[-1].cpu().numpy())


def test_non_finite_truth():
    """A NaN position gives absent rangings (mm > 0 fails); an infinite one the format's largest value."""
    N, T = 256, 3
    truth = walk(N, 0, T)[0]
    truth[1, 0, :10] = np.nan
    truth[2, 2, 10:20] = np.inf
    for fmt, top in ((L.FMT_I32_MM, 2147483647), (L.FMT_U16_MM, 65535)):
        r, _ = truth_call(N, 0, truth, fmt=fmt)
        assert (r[1, :, :10] == 0).all() and (r[2, :, 10:20] == top).all()
        assert (r[0] > 0).all() and (r[1, :, 10:] > 0).all() and (r[2, :, :10] > 0).all()
        assert (r[2, :, 20:] > 0).all() and (r[2, :, 20:] < top).all()


# ------------------------------------------------------------------------------------- 2. walk, exact cases
def test_walk_exact_cases():
    """accel_sd = 0 and hand-made states: a straight line, one reflection at each of the six walls, a reflection
    that lands beyond the opposite wall (the clamp), and the speed cap -- bit for bit against numpy."""
    import torch
    lo, hi, v_max = (0.5, 0.5, 0.0), (9.5, 9.5, 2.0), (1.5, 1.5, 0.5)
    cols = [((2.0, 3.0, 1.0), (0.3, -0.2, 0.05)),     # straight line
            ((9.45, 5.0, 1.0), (1.0, 0.0, 0.0)),      # wall x = hi
            ((0.55, 5.0, 1.0), (-1.0, 0.0, 0.0)),     # wall x = lo
            ((5.0, 9.45, 1.0), (0.0, 1.2, 0.0)),      # wall y = hi
            ((5.0, 0.52, 1.0), (0.0, -0.9, 0.0)),     # wall y = lo
            ((5.0, 5.0, 1.98), (0.0, 0.0, 0.4)),      # wall z = hi
            ((5.0, 5.0, 0.01), (0.0, 0.0, -0.3)),     # wall z = lo
            ((9.4, 5.0, 1.0), (100.0, 0.0, 0.0)),     # reflected beyond x = lo: clamped, then capped
            ((2.0, 2.0, 1.0), (3.0, -2.5, 0.9))]      # above the cap on every axis
    x = np.array([c[0] for c in cols]).T.copy()
    v = np.array([c[1] for c in cols]).T.copy()
    T = 40
    ref, xe, ve = np_walk(x, v, T, 0.1, lo, hi, v_max)
    st = torch.as_tensor(np.vstack([x, v]), device=DEV)
    tr, s, _ = walk(len(cols), 3, T, state=st, accel_sd=(0.0, 0.0, 0.0), v_max=v_max, lo=lo, hi=hi)
    assert np.array_equal(tr, ref)
    assert np.array_equal(s, np.vstack([xe, ve]))
    # each case did what it is there for
    assert np.array_equal(tr[0, :, 0], x[:, 0] + v[:, 0] * 0.1)
    assert tr[0, 0, 1] < 9.5 and tr[0, 0, 2] > 0.5 and tr[0, 1, 3] < 9.5 and tr[0, 1, 4] > 0.5
    assert tr[0, 2, 5] < 2.0 and tr[0, 2, 6] > 0.0
    assert tr[0, 0, 7] == 0.5
    assert (np.abs(np.diff(tr[:, :, 8], axis=0)) <= np.array(v_max) * 0.1 + 1e-12).all()


# -------------------------------------------------------------------------------------- 3. walk, statistics
def test_walk_statistics_and_chained_calls():
    """One-epoch calls chained through `state` (so each epoch's velocity is visible), walls and caps far away."""
    import torch
    from scipy import stats
    N, T, sd = 65536, 12, np.array([0.5, 0.3, 0.2])
    big = dict(accel_sd=tuple(sd), v_max=(INF, INF, INF), lo=(-1e4, -1e4, -1e4), hi=(1e4, 1e4, 1e4))
    whole, s_whole, x0 = walk(N, 5, T, want_x0=True, **big)
    st = torch.as_tensor(x0, device=DEV)
    xs, vs = [x0[:3]], [x0[3:]]
    for k in range(T):
        tr, s, _ = walk(N, 5 + k, 1, state=st, **big)
        assert np.array_equal(tr[0], s[:3])
        xs.append(s[:3]); vs.append(s[3:])
    xs, vs = np.stack(xs), np.stack(vs)
    # purity: the chained calls are the one call, bit for bit
    assert np.array_equal(xs[1:], whole) and np.array_equal(np.vstack([xs[-1], vs[-1]]), s_whole)
    far = (np.abs(x0[:3]) < 1e4 - 10.0).all(axis=0)
    assert far.mean() > 0.99
    dt = 0.1
    a = (vs[1:] - vs[:-1]) / dt                                   # [T][3][N]
    for i in range(3):
        ai = a[:, i, far].ravel()
        ks = stats.kstest(ai / sd[i], "norm")
        assert ks.pvalue > 1e-3, (i, ks)
    # the position recurrence with the accelerations the velocities show
    pred = (xs[:-1] + vs[:-1] * dt) + a * (dt * dt / 2)
    assert (np.abs(pred - xs[1:])[:, :, far] <= 1e-12 * np.abs(xs[1:])[:, :, far] + 1e-12).all()
    # independent across axes and epochs
    n = a[:, 0, far].size
    for i, j in ((0, 1), (0, 2), (1, 2)):
        assert abs(np.corrcoef(a[:, i, far].ravel(), a[:, j, far].ravel())[0, 1]) < 5 / np.sqrt(n)
    for i in range(3):
        assert abs(np.corrcoef(a[:-1, i, far].ravel(), a[1:, i, far].ravel())[0, 1]) < 5 / np.sqrt(n)


def test_walk_initial_state_and_region():
    from scipy import stats
    N, T = 65536, 400
    lo, hi = ROOM_WALK["lo"], ROOM_WALK["hi"]
    tr, s, x0 = walk(N, 0, T, want_x0=True)
    for i in range(2):
        ks = stats.kstest(x0[i], "uniform", args=(lo[i], hi[i] - lo[i]))
        assert ks.pvalue > 1e-3, (i, ks)
    assert not x0[3:].any()
    # z is held exactly at the centre, its velocity stays 0
    assert (x0[2] == 1.0).all() and (tr[:, 2] == 1.0).all() and (s[2] == 1.0).all() and not s[5].any()
    for i in range(2):
        assert (tr[:, i] >= lo[i]).all() and (tr[:, i] <= hi[i]).all()
        # the tag reaches every wall
        assert (tr[:, i] < lo[i] + 0.05).any() and (tr[:, i] > hi[i] - 0.05).any()
    assert (np.abs(s[3:5]) <= 1.5).all()
    # one init call gives the same walk as the initial state followed by the epochs
    tr2, s2, none = walk(N, 0, T)
    assert none is None and np.array_equal(tr2, tr) and np.array_equal(s2, s)


def test_walk_shards_and_chunks():
    import torch
    N, T = 4096, 300
    tr, s, x0 = walk(N, 11, T, want_x0=True)
    trs, ss, x0s = walk(1000, 11, T, want_x0=True, first_filter=2000)
    assert np.array_equal(trs, tr[:, :, 2000:3000]) and np.array_equal(x0s, x0[:, 2000:3000])
    st = torch.as_tensor(x0, device=DEV)
    parts = [walk(N, 11 + k0, n, state=st)[0] for k0, n in ((0, 100), (100, 1), (101, 199))]
    assert np.array_equal(np.concatenate(parts), tr)
    assert np.array_equal(st.cpu().numpy(), s)
    other = walk(N, 11, T, seed=synth.SEED + 1)[0]
    assert (other[:, :2] != tr[:, :2]).mean() > 0.9


# ------------------------------------------------------------------------------------- 4. geometry on a walk
def test_walk_mask_equals_numpy_slab_test():
    N, T = 4096, 200
    anc = synth.anchors_for(8)
    boxes = STUDY.copy()
    boxes[:, 8] = 0.0
    tr = walk(N, 0, T)[0]
    r, m = truth_call(N, 0, tr, boxes=boxes, anc=anc, sigma_r=0.0)
    blocked = np.zeros(r.shape, dtype=bool)
    for blk, _ in slab(tr, anc, boxes):
        blocked |= blk
    assert (r > 0).all()
    assert np.array_equal(m, bits(blocked))
    assert 0.01 < blocked.mean() < 0.5
    # a tag inside the pillar is blocked from every anchor
    inside = ((tr[:, 0] > boxes[0, 0]) & (tr[:, 0] < boxes[0, 3]) & (tr[:, 1] > boxes[0, 1]) & (tr[:, 1] < boxes[0, 4]))
    assert inside.any() and (m[inside] == 0xFF).all()
    # the loss draws are the documented counters
    boxes[:, 8] = 0.5
    r, m = truth_call(N, 0, tr, boxes=boxes, anc=anc, sigma_r=0.0)
    u, _ = geo_uniforms(synth.SEED, 0, N, 0, T, 8)
    keep = np.ones(r.shape)
    for b, (blk, _) in zip(boxes, slab(tr, anc, boxes)):
        keep = np.where(blk, keep * (1.0 - b[8]), keep)
    assert np.array_equal(r == 0, blocked & (u < 1.0 - keep))


# ------------------------------------------------------------------------------------------- 5. end to end
def test_toa_montecarlo_on_a_walk_whole_equals_chunked():
    from roskfpos_b200.batch import Batch
    N, T = 4096, 60
    anc = synth.anchors_for(8)
    sets = ("present", "los", "used")
    edges = np.array([0.05, 0.1, 0.2, 0.5, 1.0])
    out = []
    for chunk in (T, 25):
        with Batch(L.MODEL_T6, N, anchors=anc, accel_noise=0.5, variant=1, num_ignored_rangings=1) as b:
            out.append(synth.toa_montecarlo(b, T, chunk, anc, err=0.10, p_nlos=0.05, nlos_mean=0.8,
                                            hist=(edges, "err"), score=True, crlb=sets, obstacles=STUDY, walk=ROOM_WALK))
    (rows, h, sc, cr), (rows2, h2, sc2, cr2) = out
    assert np.array_equal(rows, rows2) and np.array_equal(h, h2) and np.array_equal(sc, sc2)
    for s in sets:
        assert np.array_equal(cr[s], cr2[s])
    assert sc[:, 2].min() > 0
    # without walk the call is the Lissajous run, with a different truth
    with Batch(L.MODEL_T6, N, anchors=anc, accel_noise=0.5, variant=1, num_ignored_rangings=1) as b:
        rows3 = synth.toa_montecarlo(b, T, T, anc, err=0.10, p_nlos=0.05, nlos_mean=0.8, obstacles=STUDY)
    assert not np.array_equal(rows3, rows)
    with pytest.raises(ValueError):
        with Batch(L.MODEL_T6, 64, anchors=anc, accel_noise=0.5) as b:
            synth.toa_montecarlo(b, 4, 4, anc, walk=dict(ROOM_WALK, tag_z=1.0))


def walk_log(N, T, m=8, **kw):
    """A walk log from the walk's x0: host (ranges [T][m][N], x0 [6][N])."""
    w = synth.walk_truth_chunk(N, 0, T, DEV, seed=synth.SEED, period=0.1, want_x0=True, **ROOM_WALK)
    r = synth.toa_montecarlo_chunk(N, 0, T, synth.anchors_for(m), DEV, truth=w["truth"], **kw)["ranges"]
    return r.cpu().numpy(), w["x0"].cpu().numpy()


@pytest.mark.parametrize("case", ["plain_m8", "loo_m16_nlos"])
def test_t6_parity_on_walk_log(kflib, oracle, case):
    """Under the tolerances of test_gpu_synth_toa's parity on the Lissajous log."""
    m, T = (16, 15) if case == "loo_m16_nlos" else (8, 20)
    N, n = 8192, 2048
    anc = synth.anchors_for(m)
    nlos = dict(p_nlos=0.15, nlos_mean=0.8) if case != "plain_m8" else {}
    r, x0 = walk_log(N, T, m=m, **nlos)
    loo = case.startswith("loo")
    got = t6_run(r, x0, anc, **({"ignore_worst_anchor": 1, "ignore_cost_threshold": 0.0} if loo else {}))
    sub = {k: got[k][..., :n] for k in ("x", "P", "status", "sel")}
    ref, per = oracle_t6(oracle, x0[:, :n], np.ascontiguousarray(r[:, :, :n]), anc,
                         **(dict(ignore_worst=True, thr=0.0) if loo else {}))
    keys = dict(float_keys=("x",), cov_keys=("P",), int_keys=("status", "sel") if loo else ("status",))
    rep = assert_parity(sub, ref, per, min_stable=0.93 if loo else 0.99, max_tie_frac=1e-3,
                        what=f"walk log {case}", **keys)
    print("parity report", case, rep)


def test_ml_variant1_on_walk_epoch(kflib, oracle):
    from roskfpos_b200.batch import Batch
    N, m = 20000, 16
    anc = synth.anchors_for(m)
    r, _ = walk_log(N, 1, m=m, p_nlos=0.15)
    r = np.ascontiguousarray(r[0])
    start = [1.0, 1.0, 4.0]
    with Batch(L.MODEL_ML, N, anchors=anc, variant=1, num_ignored_rangings=2, ml_start=start) as b:
        got = b.ml_solve(r, err=0.01)
    kw = dict(variant=1, n_ignore=2)
    ref = oracle.ml_batch(r, anc, 0.01, start, **kw)
    per = [oracle.ml_batch(p, anc, 0.01, start, **kw) for p in ulp_perturbations(to_metres(r))]
    rep = assert_parity(got, ref, per, float_keys=("pos",), int_keys=("status", "sel"), min_stable=0.98,
                        max_tie_frac=1e-3, what="ML variant 1 on a walk epoch")
    print("parity report ML", rep)


# ---------------------------------------------------------------------------------- 6. errors and the sync rule
def test_error_paths():
    import torch
    N = 256
    st = torch.zeros((6, N), dtype=torch.float64, device=DEV)
    tr = torch.zeros((4, 3, N), dtype=torch.float64, device=DEV)

    def call(T=4, **kw):
        a = dict(dict(seed=1, period=0.1, init=1, **ROOM_WALK), **kw)
        w = L.KfposSynthWalk(seed=a["seed"], period=a["period"], init=a["init"])
        w.accel_sd[:], w.v_max[:], w.lo[:], w.hi[:] = a["accel_sd"], a["v_max"], a["lo"], a["hi"]
        return L.lib().kfpos_synth_walk(0, N, T, C.byref(w), C.c_void_p(st.data_ptr()), C.c_void_p(tr.data_ptr()),
                                        None)
    assert call() == 0 and call(T=0) == 0 and call(init=0) == 0
    assert call(v_max=(INF, INF, INF), accel_sd=(0.0, 0.0, 0.0)) == 0
    for kw in (dict(T=-1), dict(period=0.0), dict(init=3), dict(accel_sd=(-1.0, 0.0, 0.0)), dict(v_max=(0.0, 1, 1)),
               dict(lo=(9.5, 0.5, 0.5)), dict(hi=(INF, 9.5, 1.5))):
        assert call(**kw) == -1, kw
    torch.cuda.synchronize()
    with pytest.raises(L.KfposError):
        synth.walk_truth_chunk(16, 0, 2, DEV, seed=1, period=0.1, accel_sd=0.5, v_max=1.0, lo=0.0, hi=0.0)
    with pytest.raises(ValueError):
        synth.walk_truth_chunk(16, 0, 2, DEV, seed=1, period=0.1, state=torch.zeros((6, 8), device=DEV,
                                                                                     dtype=torch.float64), **ROOM_WALK)
    with pytest.raises(ValueError):
        synth.toa_montecarlo_chunk(16, 0, 2, synth.anchors_for(8), DEV, truth=torch.zeros((2, 3, 8), device=DEV,
                                                                                           dtype=torch.float64))
    with pytest.raises(ValueError):
        synth.toa_montecarlo_chunk(16, 0, 2, synth.anchors_for(8), DEV, want_x0=True,
                                   truth=torch.zeros((2, 3, 16), device=DEV, dtype=torch.float64))


def test_sync_rule():
    """Device-only calls leave the work queued; a host truth, state or output is staged and the stream synchronised."""
    import torch
    from tests.test_gpu_staging import _busy_after
    N, M, T = 1 << 16, 8, 20
    s = torch.cuda.Stream()
    sp = C.c_void_p(s.cuda_stream)
    anc = np.ascontiguousarray(synth.anchors_for(M))
    gen = L.KfposSynthToa(seed=9, sigma_r=0.1)
    tbl = table(STUDY)
    w = L.KfposSynthWalk(seed=9, period=0.1, init=1)
    w.accel_sd[:], w.v_max[:], w.lo[:], w.hi[:] = ROOM_WALK["accel_sd"], ROOM_WALK["v_max"], ROOM_WALK["lo"], \
        ROOM_WALK["hi"]
    d_st = torch.empty((6, N), dtype=torch.float64, device=DEV)
    d_tr = torch.empty((T, 3, N), dtype=torch.float64, device=DEV)
    d_r = torch.empty((T, M, N), dtype=torch.int32, device=DEV)
    d_m = torch.empty((T, N), dtype=torch.int32, device=DEV)
    h_st, h_tr = np.zeros((6, N)), np.zeros((T, 3, N))
    h_r, h_m = np.zeros((T, M, N), dtype=np.int32), np.zeros((T, N), dtype=np.uint32)
    dp = lambda x: C.c_void_p(x.data_ptr())
    hp = lambda x: C.c_void_p(x.ctypes.data)

    def wk(st, tr):
        return lambda: L.check(L.lib().kfpos_synth_walk(0, N, T, C.byref(w), st, tr, sp), "walk")

    def gn(tr, r, m):
        return lambda: L.check(L.lib().kfpos_synth_toa_ranges_truth(0, N, M, hp(anc), T, tr, C.byref(gen), 3,
                                                                    C.cast(tbl, C.c_void_p), L.FMT_I32_MM, r, m, sp),
                               "truth")
    assert _busy_after(wk(dp(d_st), dp(d_tr)), s)
    assert not _busy_after(wk(hp(h_st), hp(h_tr)), s)
    assert not _busy_after(wk(dp(d_st), hp(h_tr)), s)
    assert np.array_equal(h_st, d_st.cpu().numpy()) and np.array_equal(h_tr, d_tr.cpu().numpy())
    w.init = 0  # a host state is read as well as written
    st0 = d_st.clone()
    h_st[:] = st0.cpu().numpy()
    assert not _busy_after(wk(hp(h_st), dp(d_tr)), s, warm=0)
    d_st.copy_(st0)
    wk(dp(d_st), dp(d_tr))()
    s.synchronize()
    assert np.array_equal(h_st, d_st.cpu().numpy())
    h_tr[:] = d_tr.cpu().numpy()
    assert _busy_after(gn(dp(d_tr), dp(d_r), dp(d_m)), s)
    assert _busy_after(gn(dp(d_tr), dp(d_r), None), s)
    assert not _busy_after(gn(hp(h_tr), dp(d_r), dp(d_m)), s)
    assert not _busy_after(gn(dp(d_tr), hp(h_r), hp(h_m)), s)
    assert np.array_equal(h_r, d_r.cpu().numpy()) and np.array_equal(h_m, d_m.cpu().numpy().view(np.uint32))
    torch.cuda.synchronize()
