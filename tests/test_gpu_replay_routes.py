"""GPU: every launcher route of the replay kernels (tests/replay_routes.py), with the per-epoch statistics off, on
(ES) and on with a histogram (ES + EH).  For each route:

- the profiler shows that each run launched the row's instantiation with the ES / EH flags it asked for;
- statistics off, the filter outputs agree with the CPU oracle at the bars of the existing parity tests;
- the ES and ES + EH twins reproduce the statistics-off outputs bit for bit (x, P, status, traj, sel, counters,
  the final-state error_stats);
- epoch_stats columns 0..3 equal the documented summation tree of the statistics-off trajectory, columns 4..5 the
  NEES of a step-by-step statistics-off replay; the histogram counts equal the host binning;
- the same workload with the filters in a fixed random order gives the same per-filter outputs and counts.

Then the route switches between chunks: the ML-initialisation flag that the host drops once it has seen every
filter initialised (K8 2-D mode, T9), and per-filter time steps that happen to be common."""
import json
import os
import re
import shutil
import subprocess
import tempfile
from contextlib import contextmanager

import numpy as np
import pytest

from roskfpos_b200 import synth
from tests.replay_routes import ROUTES, Route
from tests.test_gpu_epoch_stats import nees_np, terms, tree
from tests.test_gpu_error_hist import EDGES, NEES_EDGES, check_nees, err2, host_hist
from tests.util import assert_parity, to_metres, ulp_perturbations

pytestmark = pytest.mark.gpu

TAG_Z = 1.049       # K8: fixedHeight of synth.K8_XML, the z the statistics use
G = 4               # filter groups with one per-filter time-step pattern each
IMU_COV = np.array([[0.02, 0.002, 0.0], [0.002, 0.03, 0.001], [0.0, 0.001, 0.05]]).ravel()
QUANTITIES = ("err", "err_xy", "nees")


# ---------------------------------------------------------------------------------------------- kernel launches
_KERNEL = re.compile(r"\b(?:kfpos::)?((?:t6|k8|t9)_replay_kernel<[^<>]*>)")


@contextmanager
def launches():
    """Collects the names of the CUDA kernels launched inside the block (torch.profiler, CUDA activity) into the
    list it yields; fails when the profiler saw no kernel of this library at all."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    names = []
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        yield names
        torch.cuda.synchronize()
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "trace.json")
        prof.export_chrome_trace(path)
        with open(path) as f:
            trace = json.load(f)
    found = [e["name"] for e in trace.get("traceEvents", []) if e.get("cat") == "kernel"]
    mangled = [n for n in found if n.startswith("_Z")]
    if mangled and shutil.which("c++filt"):
        out = subprocess.run(["c++filt"], input="\n".join(mangled), capture_output=True, text=True).stdout
        found = [n for n in found if not n.startswith("_Z")] + out.splitlines()
    names += found
    assert any("kfpos::" in n for n in names), (
        "the profiler recorded no kfpos:: kernel: it does not see the launches of libkfpos_b200.so, so this test "
        f"cannot tell which replay kernel ran (kernels seen: {sorted(set(names))[:8]})")


def replay_kernels(names):
    return {m.group(1) for n in names for m in [_KERNEL.search(n)] if m}


# ---------------------------------------------------------------------------------------------- workloads
def workload(r: Route, N, seed):
    """Inputs of a row: dict(anc, rr (wire format), err, x0, rows (statistics truth), truth_end, events, sens, dtf,
    skip [T][N], dt [T] or None (per-filter), cfg (Batch keywords))."""
    rng = np.random.default_rng(seed)
    T = 2 if r.variant == 2 else 6
    anc = synth.anchors_for(r.m)
    zt = TAG_Z if r.model == "K8" else 1.0
    truth = synth.truth_lissajous(N, T, 0.1, seed=seed, z=zt)
    mm = synth.ranges_mm(truth[1:], anc, seed=seed + 1, p_nlos=0.2 if (r.variant or r.loo) else 0.0,
                         p_missing=0.1 if r.m >= 12 else 0.0)
    x0 = np.zeros(({"T6": 3, "K8": 8, "T9": 9}[r.model], N))
    x0[:3] = truth[0]
    if r.model == "K8":
        x0[2] = 0.0
    if r.mli:  # a quarter of the filters start uninitialised; some of them have no rangings in their first epochs
        un = rng.random(N) < 0.25
        x0[:2 if r.model == "K8" else 3, un] = np.nan
        late = np.where(un, rng.integers(0, 3, N), 0)
        for t in range(2):
            mm[t][:, late > t] = 0
    rr = {"f64": mm / 1000.0, "i32": mm.astype(np.int32), "u16": mm.astype(np.uint16)}[r.fmt]
    err = rng.uniform(0.005, 0.05, size=rr.shape) if r.pme else 0.01
    dtf, skip, dt = None, np.zeros((T, N), dtype=bool), np.full(T, 0.1)
    if r.dtf:  # G interleaved groups of filters, each with its own time steps and skipped epochs
        pat_dt = rng.uniform(0.05, 0.15, size=(T, G))
        pat_skip = rng.random((T, G)) < 0.3
        pat_skip[0] = False
        g = np.arange(N) % G
        dtf = np.where(pat_skip[:, g], -1.0, pat_dt[:, g])
        skip = pat_skip[:, g]
        dt = None
    events, sens = None, None
    if r.model != "T6":
        if r.imu:
            sens = rng.normal(0, 0.2, size=(3 * T, N))
            events = []
            for t in range(T):
                events += [(synth.EV_IMU, 0.04, 3 * t, IMU_COV), (synth.EV_TOA, 0.06, t * r.m, None)]
        else:
            events = [(synth.EV_TOA, 0.1, t * r.m, None) for t in range(T)]
    rows = truth[1:].copy()
    if r.model == "K8":
        rows[:, 2] = TAG_Z
    cfg = dict(accel_noise=0.5)
    if r.model != "T6":
        cfg["jolt"] = 0.5
    if r.model == "K8":
        cfg["xml"] = synth.K8_XML
    if r.loo:
        cfg.update(ignore_worst_anchor=1, ignore_cost_threshold=0.0)
    if r.variant:
        cfg.update(variant=r.variant, num_ignored_rangings=2 if r.variant == 1 else 0)
    if r.mli:
        cfg["ml_initial_position"] = 1
        if r.model == "K8":
            cfg["use_fixed_height"] = 1
    if r.zero_tz:
        cfg["ml2d_zero_tentative_z"] = 1
    return dict(anc=anc, rr=rr, err=err, x0=x0, rows=rows, truth_end=truth[-1].copy(), events=events, sens=sens,
                dtf=dtf, skip=skip, dt=dt, cfg=cfg, T=T)


def permuted(w, perm):
    """The workload with filter perm[i] in position i."""
    p = dict(w)
    for k in ("rr", "x0", "rows", "truth_end", "sens", "dtf", "skip"):
        if p[k] is not None:
            p[k] = np.ascontiguousarray(p[k][..., perm])
    if not np.isscalar(w["err"]):
        p["err"] = np.ascontiguousarray(w["err"][..., perm])
    return p


def model_id(kflib, r):
    return {"T6": kflib.MODEL_T6, "K8": kflib.MODEL_K8, "T9": kflib.MODEL_T9}[r.model]


def replay(b, r, w):
    """One replay launch of the whole workload: (traj, sel or None)."""
    if r.dtf:
        return b.replay_epochs(w["dtf"], w["rr"], err=w["err"], want_traj=True), None
    if r.model == "T6":
        return b.replay_toa(w["dt"], w["rr"], err=w["err"], want_traj=True, want_sel=True)
    return b.replay_events(w["events"], ranges=w["rr"], sensors=w["sens"], err=w["err"], want_traj=True), None


def run_gpu(kflib, r, w, stats=None, quantity=None):
    """stats None / "es" / "eh": the outputs of one replay and the replay kernels it launched."""
    from roskfpos_b200.batch import Batch
    N = w["x0"].shape[-1]
    with Batch(model_id(kflib, r), N, anchors=w["anc"], **w["cfg"]) as b:
        if stats:
            b.set_truth_traj(w["rows"])
        if stats == "eh":
            b.set_error_hist(NEES_EDGES if quantity == "nees" else EDGES, quantity)
        b.set_truth(w["truth_end"])
        b.set_state(w["x0"])
        with launches() as names:
            traj, sel = replay(b, r, w)
        x, P, st = b.get_state()
        out = dict(x=x, P=P, st=st, traj=traj, sel=sel, cnt=b.counters(), fin=b.error_stats(),
                   kernels=replay_kernels(names))
        if stats:
            out["es"] = b.epoch_stats()
        if stats == "eh":
            out["hist"] = b.error_hist()
    return out


# ---------------------------------------------------------------------------------------------- the oracle
def oracle_run(oracle, r, w, rr):
    """The oracle on the range log `rr` (any wire format): dict(x, P, status[, sel]) over all filters.  Per-filter
    time steps: once per group of filters, on that group's own epochs."""
    N = w["x0"].shape[-1]
    if not r.dtf:
        return _oracle(oracle, r, w, rr, w["err"], w["x0"], w["dt"], w["events"], w["sens"])
    out = None
    for g in range(G):
        idx = np.arange(g, N, G)
        keep = ~w["skip"][:, g]
        dt = w["dtf"][keep, g]
        err = w["err"] if np.isscalar(w["err"]) else np.ascontiguousarray(w["err"][keep][..., idx])
        events = [(synth.EV_TOA, float(d), k * r.m, None) for k, d in enumerate(dt)] if r.model != "T6" else None
        o = _oracle(oracle, r, w, np.ascontiguousarray(rr[keep][..., idx]), err, w["x0"][:, idx], dt, events, None)
        o.pop("sel", None)  # replay_epochs has no selection output
        if out is None:
            out = {k: np.zeros(v.shape[:-1] + (N,), dtype=v.dtype) for k, v in o.items()}
        for k, v in o.items():
            out[k][..., idx] = v
    return out


def _oracle(oracle, r, w, rr, err, x0, dt, events, sens):
    if r.model == "T6":
        o = oracle.t6_replay(x0, None, rr, w["anc"], dt, err, ignore_worst=r.loo, thr=0.0, variant=r.variant,
                             n_ignore=2 if r.variant == 1 else 0)
        return dict(x=o["x"], P=o["P"], status=o["status"], sel=o["sel"])
    if r.model == "K8":
        ocfg = dict(synth.K8_ORACLE_CFG, variant=r.variant, n_ignore=2 if r.variant == 1 else 0)
        if r.mli:
            ocfg.update(ml_init=1, use_fixed_height=1)
        o = oracle.k8_replay(x0, None, events, rr, sens, w["anc"], err, oracle.k8_cfg(0.5, 0.5, **ocfg),
                             b1_zero_z=r.zero_tz)
    else:
        o = oracle.t9_events(x0, None, events, rr, sens, w["anc"], err, variant=r.variant,
                             n_ignore=2 if r.variant == 1 else 0, ml_init=int(r.mli))
    return dict(x=o["x"], P=o["P"], status=o["status"])


def status_mask(r):
    """Status bits compared with the oracle: the same as the existing parity tests of the model."""
    m = {"T6": ~32, "K8": ~(32 | 64), "T9": ~0}[r.model]
    return m & ~256 if r.mli else m


def check_oracle(oracle, r, w, got):
    """Statistics off against the oracle, with the stability rule and the bars of the existing tests of the mode:
    test_gpu_fuzz for T6, test_gpu_k8 / test_gpu_t9 for the variants, test_gpu_ml_init for ML initialisation;
    every filter for the remaining K8 / T9 routes (test_gpu_fuzz, test_gpu_t9)."""
    ref = oracle_run(oracle, r, w, w["rr"])
    mask = status_mask(r)
    n = 3 if r.model == "T6" else len(ref["x"])
    g = dict(x=got["x"][:n], P=got["P"], status=got["st"] & mask)
    ints = ("status",)
    if "sel" in ref and got["sel"] is not None:
        g["sel"] = got["sel"]
        ints = ("status", "sel")
    if r.model == "T6":
        few = r.m <= 5 or r.variant or r.loo
        n_random, min_stable = (32 if r.variant else 8), (0.4 if few else 0.85)
    elif r.variant:
        n_random = 12
        min_stable = 0.9 if r.variant == 1 else (0.6 if r.model == "K8" else 0.4)
    elif r.mli:
        n_random, min_stable = 2, (0.85 if r.model == "K8" else 0.98)
    else:
        n_random, min_stable = None, 1.0
    per = [] if n_random is None else [oracle_run(oracle, r, w, p)
                                       for p in ulp_perturbations(to_metres(w["rr"]), n_random=n_random)]
    for d in [ref] + per:
        d["status"] = d["status"] & mask
    assert_parity(g, ref, per, float_keys=("x",), cov_keys=("P",), int_keys=ints, min_stable=min_stable,
                  max_tie_frac=1e-3, what=f"route {r.id}")


# ---------------------------------------------------------------------------------------------- host statistics
def step_reference(kflib, r, w):
    """Replays the workload epoch by epoch with the statistics off, restoring (x, P) -- and the latched sensor
    samples of an IMU schedule -- before each epoch: per row (status != 0, NEES, counted) from the state after it."""
    from roskfpos_b200.batch import Batch
    N, T = w["x0"].shape[-1], w["T"]
    nd = 2 if r.model == "K8" else 3
    err = w["err"]
    chunks = []
    if r.model != "T6" and not r.dtf:  # the event schedule cut after every ranging event
        cur = []
        for ev in w["events"]:
            cur.append(ev)
            if ev[0] == synth.EV_TOA:
                chunks.append(cur)
                cur = []
    bad, nees, cnt = [], [], []
    with Batch(model_id(kflib, r), N, anchors=w["anc"], **w["cfg"]) as b:
        b.set_state(w["x0"])
        for t in range(T):
            if t:
                b.set_state(x, P)
                if r.imu:
                    b.set_latches(*lat)
            e_t = err if np.isscalar(err) else np.ascontiguousarray(err[t:t + 1])
            if r.dtf:
                b.replay_epochs(np.ascontiguousarray(w["dtf"][t:t + 1]), np.ascontiguousarray(w["rr"][t:t + 1]), err=e_t)
            elif r.model == "T6":
                b.replay_toa(w["dt"][t:t + 1], np.ascontiguousarray(w["rr"][t:t + 1]), err=e_t)
            else:
                b.replay_events(chunks[t], ranges=w["rr"], sensors=w["sens"], err=err)
            x, P, st = b.get_state()
            if r.imu:
                lat = b.get_latches()
            Pf = P.reshape(b.n, b.n, N).transpose(2, 0, 1)
            pz = np.full(N, TAG_Z) if r.model == "K8" else x[2]
            v, ok = nees_np(np.stack([x[0], x[1], pz], axis=1) - w["rows"][t].T, Pf, nd)
            sk = w["skip"][t]
            bad.append((st != 0) & ~sk)
            nees.append(np.where(sk, 0.0, v))
            cnt.append(ok & ~sk)
    return np.array(bad), np.array(nees), np.array(cnt)


def stats_traj(r, traj):
    """traj as the statistics see it: K8 row 2 is the heading, the statistics use the tag height."""
    tr = traj.copy()
    if r.model == "K8":
        tr[:, 2] = TAG_Z
    return tr


def check_stats(r, w, off, es, hists, ref):
    bad, nees, cnt = ref
    v = terms(stats_traj(r, off["traj"]), w["rows"], skip=w["skip"])
    assert np.array_equal(es[:, :4], tree(np.concatenate([v, bad[..., None] * 1.0], axis=-1))), "columns 0..3"
    ref_n = tree(np.stack([nees, cnt * 1.0], axis=-1))
    assert np.array_equal(es[:, 5], ref_n[:, 1]), "column 5"
    assert np.allclose(es[:, 4], ref_n[:, 0], rtol=1e-12, atol=0), "column 4"
    assert (es[:, 2] > 0).all()
    e2, exy, fin = err2(stats_traj(r, off["traj"]), w["rows"])
    fin = fin & ~w["skip"]
    assert np.array_equal(hists["err"], host_hist(e2, fin, EDGES * EDGES)), "err histogram"
    assert np.array_equal(hists["err_xy"], host_hist(exy, fin, EDGES * EDGES)), "err_xy histogram"
    assert np.array_equal(hists["nees"].sum(axis=1), cnt.sum(axis=1).astype(np.uint64))
    check_nees(hists["nees"], nees, cnt)


# ---------------------------------------------------------------------------------------------- per route
SAME = ("x", "P", "st", "traj", "sel", "fin")


def assert_same(a, b, what):
    for k in SAME:
        if a[k] is None:
            assert b[k] is None, (what, k)
            continue
        assert np.array_equal(a[k], b[k], equal_nan=np.asarray(a[k]).dtype.kind == "f"), (what, k)
    assert a["cnt"] == b["cnt"], what


def route_params():
    out = []
    for r in ROUTES:
        for N in ((129, 1000) if r.big else (129,)):
            out.append(pytest.param(r, N, id=f"{r.id}-N{N}"))
    return out


@pytest.mark.parametrize("r,N", route_params())
def test_route(kflib, oracle, r, N):
    seed = 100 + ROUTES.index(r)
    w = workload(r, N, seed)
    off = run_gpu(kflib, r, w)
    assert off["kernels"] == {r.symbol(False, False)}, off["kernels"]
    check_oracle(oracle, r, w, off)

    es = run_gpu(kflib, r, w, "es")
    assert es["kernels"] == {r.symbol(True, False)}, es["kernels"]
    assert_same(off, es, "ES")
    hists = {}
    for q in QUANTITIES:
        eh = run_gpu(kflib, r, w, "eh", q)
        assert eh["kernels"] == {r.symbol(True, True)}, eh["kernels"]
        assert_same(off, eh, f"ES + EH {q}")
        assert np.array_equal(eh["es"], es["es"]), q
        hists[q] = eh["hist"]
    check_stats(r, w, off, es["es"], hists, step_reference(kflib, r, w))

    # the filters in a fixed random order: lane and warp composition must not matter
    perm = np.random.default_rng(seed + 7).permutation(N)
    inv = np.argsort(perm)
    p = run_gpu(kflib, r, permuted(w, perm), "eh", "nees")
    for k in ("x", "P", "st", "traj", "sel"):
        if off[k] is not None:
            assert np.array_equal(p[k][..., inv], off[k], equal_nan=off[k].dtype.kind == "f"), k
    assert np.array_equal(p["hist"], hists["nees"])
    assert np.array_equal(p["es"][:, [2, 3, 5]], es["es"][:, [2, 3, 5]])
    assert np.allclose(p["es"], es["es"], rtol=1e-12, atol=0)
    assert np.allclose(p["fin"], off["fin"], rtol=1e-12, atol=0) and p["fin"][2:].tolist() == off["fin"][2:].tolist()
    assert p["cnt"] == off["cnt"]


# ---------------------------------------------------------------------------------------------- route switches
def _sym(model, tup, es=False, eh=False):
    return Route(model, tup).symbol(es, eh)


@pytest.mark.parametrize("model", ["K8", "T9"])
def test_ml_init_switch(kflib, model):
    """ml_initial_position: once a launch has ended with every filter initialised and the host has seen it (here
    get_state waits), the next chunk runs the flag-free instantiation (path A).  set_state + set_latches with the
    same values re-arms the flag, and the same chunk runs the initialising instantiation (path B).  Which one runs
    depends on host timing in a real run, so chunk 2 must come out the same, bit for bit.  K8 in 2-D mode at 8
    anchors (MT = 8 on both paths); T9 at 6 anchors with accelerometer events (MT = 0 and IMU on both paths)."""
    from roskfpos_b200.batch import Batch
    N, T1, T = 1000, 3, 7
    m = 8 if model == "K8" else 6
    anc = synth.anchors_for(m)
    rng = np.random.default_rng(401)
    truth = synth.truth_lissajous(N, T, 0.1, seed=402, z=TAG_Z if model == "K8" else 1.0)
    rr = synth.ranges_mm(truth[1:], anc, seed=403).astype(np.int32)
    x0 = np.zeros((8 if model == "K8" else 9, N))
    x0[:3] = truth[0]
    un = rng.random(N) < 0.5
    rr[0][:, un & (rng.random(N) < 0.3)] = 0  # some of the uninitialised filters have no rangings in epoch 1
    if model == "K8":
        x0[2] = 0.0
        x0[:2, un] = np.nan
        cfg = dict(xml=synth.K8_XML, accel_noise=0.5, jolt=0.5, use_fixed_height=1, ml_initial_position=1)
        sens = None
        ev = [(synth.EV_TOA, 0.1, t * m, None) for t in range(T)]
        cut = T1
    else:
        x0[:3, un] = np.nan
        cfg = dict(accel_noise=0.5, jolt=0.5, ml_initial_position=1)
        sens = rng.normal(0, 0.2, size=(3 * T, N))
        ev = []
        for t in range(T):
            ev += [(synth.EV_IMU, 0.04, 3 * t, IMU_COV), (synth.EV_TOA, 0.06, t * m, None)]
        cut = 2 * T1
    mdl = kflib.MODEL_K8 if model == "K8" else kflib.MODEL_T9
    outs = {}
    for path in ("A", "B"):
        with Batch(mdl, N, anchors=anc, **cfg) as b:
            b.set_state(x0)
            b.replay_events(ev[:cut], ranges=rr, sensors=sens, err=0.01)
            x1, P1, st1 = b.get_state()
            assert not np.isnan(x1[:2]).any()
            if path == "B":
                lat = b.get_latches()
                b.set_state(x1, P1)
                b.set_latches(*lat)
            with launches() as names:
                traj = b.replay_events(ev[cut:], ranges=rr, sensors=sens, err=0.01, want_traj=True)
            x, P, st = b.get_state()
            outs[path] = dict(traj=traj, x=x, P=P, st=st if path == "A" else st | st1, lat=b.get_latches()[0],
                              kernels=replay_kernels(names))
    a, b_ = outs["A"], outs["B"]
    if model == "K8":
        assert a["kernels"] == {_sym("K8", (False, 8, False, False))}, a["kernels"]
        assert b_["kernels"] == {_sym("K8", (False, 8, False, True))}, b_["kernels"]
    else:
        assert a["kernels"] == {_sym("T9", (False, 0, True, False))}, a["kernels"]
        assert b_["kernels"] == {_sym("T9", (False, 0, True, True))}, b_["kernels"]
    for k in ("traj", "x", "P", "st", "lat"):
        assert np.array_equal(a[k], b_[k]), k


@pytest.mark.parametrize("m", [8, 16])
def test_t6_common_per_filter_dt(kflib, m):
    """T6: replay_epochs with dt_f[t][f] = dt[t] runs the FMT = -1 kernel, replay_toa the tuned one of the same
    anchor count; both do the same arithmetic, so the results are bit-identical."""
    from roskfpos_b200.batch import Batch
    N, T = 1000, 6
    anc = synth.anchors_for(m)
    truth = synth.truth_lissajous(N, T, 0.1, seed=501)
    rr = synth.ranges_mm(truth[1:], anc, seed=502).astype(np.int32)
    dt = np.random.default_rng(503).uniform(0.05, 0.15, T)
    outs = []
    for per_filter in (False, True):
        with Batch(kflib.MODEL_T6, N, anchors=anc, accel_noise=0.5) as b:
            b.set_state(truth[0])
            with launches() as names:
                if per_filter:
                    traj = b.replay_epochs(np.repeat(dt[:, None], N, axis=1), rr, err=0.01, want_traj=True)
                else:
                    traj, _ = b.replay_toa(dt, rr, err=0.01, want_traj=True)
            x, P, st = b.get_state()
            outs.append(dict(traj=traj, x=x, P=P, st=st, cnt=b.counters(), kernels=replay_kernels(names)))
    assert outs[0]["kernels"] == {_sym("T6", (False, False, m, False, 1))}
    assert outs[1]["kernels"] == {_sym("T6", (False, False, m, False, -1))}
    for k in ("traj", "x", "P", "st"):
        assert np.array_equal(outs[0][k], outs[1][k]), k
    assert outs[0]["cnt"] == outs[1]["cnt"]


@pytest.mark.parametrize("model", ["K8", "T9"])
def test_event_common_per_filter_dt(kflib, oracle, model):
    """K8 / T9 at 8 anchors: per-filter time steps that are the same for every filter run the general
    instantiation (MT = 0), the common time step a tuned one (MT = 8) -- replay_epochs against replay_toa, and
    replay_events(dt_per_filter=...) against replay_events on a schedule with accelerometer events.  Both agree
    with the oracle.  The two instantiations differ in MT, yet on one NVIDIA B200 they gave the same bits for all
    four pairs (traj, x, P), so a batch does not change its results when its time steps become per filter; that
    is asserted too."""
    from roskfpos_b200.batch import Batch
    N, T, m = 1000, 6, 8
    anc = synth.anchors_for(m)
    truth = synth.truth_lissajous(N, T, 0.1, seed=601, z=TAG_Z if model == "K8" else 1.0)
    rr = synth.ranges_mm(truth[1:], anc, seed=602).astype(np.int32)
    rng = np.random.default_rng(603)
    dt = rng.uniform(0.05, 0.15, T)
    x0 = np.zeros((8 if model == "K8" else 9, N)); x0[:3] = truth[0]
    cfg = dict(accel_noise=0.5, jolt=0.5)
    aux = synth.IMU_AUX if model == "K8" else IMU_COV
    sens = rng.normal(0, 0.2, size=(3 * T, N))
    ev_toa = [(synth.EV_TOA, float(dt[t]), t * m, None) for t in range(T)]
    ev_imu = []
    for t in range(T):
        ev_imu += [(synth.EV_IMU, 0.04, 3 * t, aux), (synth.EV_TOA, float(dt[t]), t * m, None)]
    if model == "K8":
        x0[2] = 0.0
        cfg["xml"] = synth.K8_XML
        kcfg = oracle.k8_cfg(0.5, 0.5, **synth.K8_ORACLE_CFG)
        ref = lambda ev, s: oracle.k8_replay(x0, None, ev, rr, s, anc, 0.01, kcfg)
    else:
        ref = lambda ev, s: oracle.t9_events(x0, None, ev, rr, s, anc, 0.01)
    mdl = kflib.MODEL_K8 if model == "K8" else kflib.MODEL_T9
    general = _sym(model, (False, 0, True, True))

    def run(kind):
        with Batch(mdl, N, anchors=anc, **cfg) as b:
            b.set_state(x0)
            with launches() as names:
                if kind == "replay_toa":
                    traj, _ = b.replay_toa(dt, rr, err=0.01, want_traj=True)
                elif kind == "replay_epochs":
                    traj = b.replay_epochs(np.repeat(dt[:, None], N, axis=1), rr, err=0.01, want_traj=True)
                elif kind == "replay_events":
                    traj = b.replay_events(ev_imu, ranges=rr, sensors=sens, err=0.01, want_traj=True)
                else:
                    dtf = np.repeat(np.array([e[1] for e in ev_imu])[:, None], N, axis=1)
                    traj = b.replay_events(ev_imu, ranges=rr, sensors=sens, err=0.01, want_traj=True,
                                           dt_per_filter=dtf)
            x, P, st = b.get_state()
            return dict(traj=traj, x=x, P=P, st=st, kernels=replay_kernels(names))
    cases = [("replay_toa", "replay_epochs", ref(ev_toa, None), _sym(model, (False, 8, False, False))),
             ("replay_events", "replay_events_ragged", ref(ev_imu, sens),
              _sym(model, (False, 8, False, False) if model == "K8" else (False, 8, True, False)))]
    for common, per_filter, o, tuned in cases:
        a, b_ = run(common), run(per_filter)
        assert a["kernels"] == {tuned}, a["kernels"]
        assert b_["kernels"] == {general}, b_["kernels"]
        for g in (a, b_):
            assert_parity(dict(x=g["x"], P=g["P"]), o, [], float_keys=("x",), cov_keys=("P",),
                          what=f"{model} {common} / {per_filter}")
        for k in ("traj", "x", "P", "st"):
            assert np.array_equal(a[k], b_[k]), (common, per_filter, k)
