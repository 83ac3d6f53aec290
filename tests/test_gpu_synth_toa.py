"""The device-side ranging generator (kfpos_synth_toa_ranges, synth.toa_montecarlo_chunk / toa_montecarlo):
a pure function of (seed, filter, epoch, anchor) with the documented Philox counters, the documented noise,
dropout and NLOS statistics, and a log that drives every ranging consumer as a stored log does."""
import ctypes as C

import numpy as np
import pytest

from roskfpos_b200 import lib as L, synth
from tests.util import assert_parity, to_metres, ulp_perturbations

pytestmark = pytest.mark.gpu

DEV = "cuda:0"


def gen(n, epoch0, T, m=8, **kw):
    """Host copies of a generated chunk: ranges [T][M][N] and the truth [T][3][N]."""
    w = synth.toa_montecarlo_chunk(n, epoch0, T, synth.anchors_for(m), DEV, want_truth=True, want_x0=True, **kw)
    return w["ranges"].cpu().numpy(), w["truth"].cpu().numpy(), w["x0"].cpu().numpy()


def distances_mm(truth, anc):
    """Host distances [T][M][N] in mm from the device truth."""
    return np.sqrt(((truth[:, None, :, :] - anc[None, :, :, None]) ** 2).sum(axis=2)) * 1000.0


# ------------------------------------------------------------------ numpy Philox4x32-10 (integer-only, exact)
M32 = np.uint64(0xFFFFFFFF)


def philox(c0, c1, c2, c3, k0, k1):
    c = [np.asarray(v, dtype=np.uint64) & M32 for v in np.broadcast_arrays(c0, c1, c2, c3)]
    k0, k1 = np.uint64(k0), np.uint64(k1)
    for _ in range(10):
        p0 = np.uint64(0xD2511F53) * c[0]
        p1 = np.uint64(0xCD9E8D57) * c[2]
        c = [(p1 >> np.uint64(32)) ^ c[1] ^ k0, p1 & M32, (p0 >> np.uint64(32)) ^ c[3] ^ k1, p0 & M32]
        k0, k1 = (k0 + np.uint64(0x9E3779B9)) & M32, (k1 + np.uint64(0xBB67AE85)) & M32
    return c


def uniform2(c):
    a = (c[0] << np.uint64(32)) | c[1]
    b = (c[2] << np.uint64(32)) | c[3]
    s = 1.0 / 9007199254740992.0
    return ((a >> np.uint64(11)).astype(np.float64) + 0.5) * s, ((b >> np.uint64(11)).astype(np.float64) + 0.5) * s


def impairment_uniforms(seed, first_filter, N, epoch0, T, M):
    """(u, v) [T][M][N] of the counters (gf lo, gf hi, g, 0x80000000 | a), key (seed lo, seed hi)."""
    gf = np.uint64(first_filter) + np.arange(N, dtype=np.uint64)
    g = (np.uint64(epoch0) + np.arange(T, dtype=np.uint64))[:, None, None]
    a = (np.uint64(0x80000000) | np.arange(M, dtype=np.uint64))[None, :, None]
    c = philox((gf & M32)[None, None, :], (gf >> np.uint64(32))[None, None, :], g, a,
               seed & 0xFFFFFFFF, seed >> 32)
    return uniform2([np.broadcast_to(v, (T, M, N)) for v in c])


# ------------------------------------------------------------------------------------------------ 1. purity
def test_pure_function_of_seed_filter_epoch_anchor():
    kw = dict(sigma_r=0.1, p_missing=0.1, p_nlos=0.1)
    full, truth, _ = gen(4096, 0, 12, **kw)
    shard, _, _ = gen(500, 0, 12, first_filter=1000, **kw)
    assert np.array_equal(shard, full[:, :, 1000:1500])
    part, tpart, _ = gen(4096, 3, 4, **kw)
    assert np.array_equal(part, full[3:7])
    assert np.array_equal(tpart, truth[3:7])
    other, _, _ = gen(4096, 0, 12, seed=synth.SEED + 1, **kw)
    assert (other != full).mean() > 0.9
    u16, _, _ = gen(4096, 0, 12, fmt=L.FMT_U16_MM, **kw)
    assert u16.dtype == np.uint16
    assert np.array_equal(u16.astype(np.int32), np.minimum(full, 65535))
    # far anchors: uint16 clamps at 65535 where int32 keeps the value
    anc = synth.anchors_for(8) + np.array([70.0, 0.0, 0.0])
    w32 = synth.toa_montecarlo_chunk(256, 0, 2, anc, DEV)["ranges"].cpu().numpy()
    w16 = synth.toa_montecarlo_chunk(256, 0, 2, anc, DEV, fmt=L.FMT_U16_MM)["ranges"].cpu().numpy()
    assert (w32 > 65535).any() and (w32 < 65535).any()
    assert np.array_equal(w16.astype(np.int64), np.minimum(w32, 65535))


def test_chunk_beyond_one_launch():
    """More epochs than one launch carries (1024): the times of every launch are the right ones."""
    r, _, _ = gen(256, 0, 2100)
    tail, _, _ = gen(256, 2000, 100)
    assert np.array_equal(r[2000:], tail)


# ------------------------------------------------------------------------------------ 2. counter layout
def test_counter_layout_matches_numpy_philox():
    N, T, M, epoch0, ff, seed = 3000, 7, 8, 41, 123456789012, 0x1234567890ABCDEF
    anc = synth.anchors_for(M)
    w = synth.toa_montecarlo_chunk(N, epoch0, T, anc, DEV, seed=seed, sigma_r=0.0, p_missing=0.3,
                                   first_filter=ff, want_truth=True)
    r = w["ranges"].cpu().numpy()
    u, v = impairment_uniforms(seed, ff, N, epoch0, T, M)
    assert np.array_equal(r == 0, u < 0.3)  # bit for bit: Philox is integer-only
    # no noise: the present rangings are the floored distances
    d = distances_mm(w["truth"].cpu().numpy(), anc)
    ok = r > 0
    assert np.abs(r[ok] - np.floor(d[ok])).max() <= 1
    # NLOS: the bias of the documented draw, -nlos_mean log(v / p_nlos) where v < p_nlos
    w = synth.toa_montecarlo_chunk(N, epoch0, T, anc, DEV, seed=seed, sigma_r=0.0, p_nlos=0.25, nlos_mean=0.5,
                                   first_filter=ff)
    r = w["ranges"].cpu().numpy()
    with np.errstate(divide="ignore"):
        bias = np.where(v < 0.25, -0.5 * np.log(v / 0.25), 0.0)
    assert np.abs(r - np.floor(d + bias * 1000.0)).max() <= 1


# ------------------------------------------------------------------------------------------- 3. statistics
def test_noise_dropout_and_nlos_statistics():
    from scipy import stats
    N, T, M = 131072, 10, 8
    anc = synth.anchors_for(M)
    # LOS: mm - 1000 d = 1000 sigma n + (floor(x) - x): mean -0.5 mm, variance (1000 sigma)^2 + 1/12 mm^2
    sigma = 0.01
    r, truth, _ = gen(N, 0, T, sigma_r=sigma)
    res = r - distances_mm(truth, anc)
    n = res.size
    sd = np.sqrt((1000 * sigma) ** 2 + 1 / 12)
    assert abs(res.mean() + 0.5) < 5 * sd / np.sqrt(n)
    assert abs(res.std() - sd) < 5 * sd / np.sqrt(2 * n)
    assert abs(stats.kurtosis(res.ravel())) < 0.02  # Gaussian
    # impairments, no noise: a missing ranging is 0; an LOS one lies in (d - 1 mm, d]; an NLOS one above d
    pm, pn, mean = 0.1, 0.2, 0.8
    r, truth, _ = gen(N, 100, T, sigma_r=0.0, p_missing=pm, p_nlos=pn, nlos_mean=mean)
    d = distances_mm(truth, anc)
    miss = r == 0
    assert abs(miss.mean() - pm) < 5 * np.sqrt(pm * (1 - pm) / n)
    ex = (r - d)[~miss]  # mm
    nlos = ex > 0
    # an NLOS bias below the flooring step (< 1 mm, probability ~ 0.5 / 800) is counted as LOS
    assert abs(nlos.mean() - pn) < 5 * np.sqrt(pn * (1 - pn) / nlos.size) + 2e-4
    assert ex[~nlos].min() > -1.0
    # the bias is exponential with mean nlos_mean: by memorylessness, b - 2 mm given b > 2 mm is too
    b = (ex[ex > 2.0] + 0.5 - 2.0) / 1000.0  # + 0.5: centre of the flooring step
    b = np.random.default_rng(5).choice(b, 50000, replace=False)
    ks = stats.kstest(b, "expon", args=(0.0, mean))
    assert ks.pvalue > 1e-3, ks
    assert abs(b.mean() - mean) < 5 * mean / np.sqrt(b.size)


# ---------------------------------------------------------------------------- 4. replay like a stored log
def t6_run(ranges, x0, anc, **cfg):
    from roskfpos_b200.batch import Batch
    N = ranges.shape[-1]
    with Batch(L.MODEL_T6, N, anchors=anc, accel_noise=0.5, **cfg) as b:
        b.set_state(x0)
        traj, sel = b.replay_toa(0.1, ranges, err=0.01, want_traj=True, want_sel=True)
        x, P, st = b.get_state()
        cnt = b.counters()
    return dict(x=x[:3], xfull=x, P=P, status=st & ~32, traj=traj, sel=sel, counters=cnt)


def test_device_log_equals_host_log():
    """The same generated ranges from the device tensor and from a host copy (the chunked host-to-device path)
    give identical state, covariance, status, trajectory, selections and counters."""
    N, T, m = 65536, 30, 8
    anc = synth.anchors_for(m)
    w = synth.toa_montecarlo_chunk(N, 0, T, anc, DEV, p_nlos=0.05, p_missing=0.05, want_x0=True)
    a = t6_run(w["ranges"], w["x0"], anc, ignore_worst_anchor=1)
    b = t6_run(w["ranges"].cpu().numpy(), w["x0"].cpu().numpy(), anc, ignore_worst_anchor=1)
    for k in ("xfull", "P", "status", "traj", "sel"):
        assert np.array_equal(a[k], b[k]), k
    assert a["counters"] == b["counters"]


def oracle_t6(oracle, x0, r, anc, n_random=4, **kw):
    def run(rr):
        out = oracle.t6_replay(x0[:3], None, rr, anc, 0.1, 0.01, **kw)
        out["status"] = out["status"] & ~32
        return out
    return run(r), [run(p) for p in ulp_perturbations(to_metres(r), n_random=n_random)]


@pytest.mark.parametrize("case", ["plain_m8", "loo_m16_nlos", "variant1_m8_nlos"])
def test_t6_parity_on_generated_log(kflib, oracle, case):
    m, T = (16, 15) if case == "loo_m16_nlos" else (8, 20)
    nlos = dict(p_nlos=0.15, nlos_mean=0.8) if case != "plain_m8" else {}
    N = 8192
    anc = synth.anchors_for(m)
    r, _, x0 = gen(N, 0, T, m=m, **nlos)
    got = t6_run(r, x0, anc, **({"ignore_worst_anchor": 1, "ignore_cost_threshold": 0.0} if case.startswith("loo") else
                                {"variant": 1, "num_ignored_rangings": 3} if case.startswith("variant1") else {}))
    n = 2048  # the oracle runs on a sample: filters are independent
    sub = {k: got[k][..., :n] for k in ("x", "P", "status", "sel")}
    kw = (dict(ignore_worst=True, thr=0.0) if case.startswith("loo") else
          dict(variant=1, n_ignore=3) if case.startswith("variant1") else {})
    ref, per = oracle_t6(oracle, x0[:, :n], np.ascontiguousarray(r[:, :, :n]), anc,
                         n_random=12 if case.startswith("variant1") else 4, **kw)
    keys = dict(float_keys=("x",), cov_keys=("P",), int_keys=("status",) if case == "plain_m8" else ("status", "sel"))
    min_stable = {"plain_m8": 0.99, "loo_m16_nlos": 0.93, "variant1_m8_nlos": 0.9}[case]
    rep = assert_parity(sub, ref, per, min_stable=min_stable, max_tie_frac=1e-3, what=f"generated log {case}", **keys)
    print("parity report", case, rep)
    assert got["counters"]["updates"] == N * T
    if nlos:
        assert (ref["sel"] >= 0).any() if case.startswith("loo") else True


def test_ml_variant1_on_generated_epoch(kflib, oracle):
    from roskfpos_b200.batch import Batch
    N, m = 20000, 16
    anc = synth.anchors_for(m)
    r, _, _ = gen(N, 0, 1, m=m, p_nlos=0.15)
    r = np.ascontiguousarray(r[0])
    start = [1.0, 1.0, 4.0]
    with Batch(L.MODEL_ML, N, anchors=anc, variant=1, num_ignored_rangings=2, ml_start=start) as b:
        got = b.ml_solve(r, err=0.01)
    kw = dict(variant=1, n_ignore=2)
    ref = oracle.ml_batch(r, anc, 0.01, start, **kw)
    per = [oracle.ml_batch(p, anc, 0.01, start, **kw) for p in ulp_perturbations(to_metres(r))]
    rep = assert_parity(got, ref, per, float_keys=("pos",), int_keys=("status", "sel"), min_stable=0.98,
                        max_tie_frac=1e-3, what="ML variant 1 on a generated epoch")
    print("parity report ML", rep)


# ----------------------------------------------------------------------------------- 5. toa_montecarlo
def test_toa_montecarlo_chunking_and_sharding():
    from roskfpos_b200.batch import Batch, epoch_summary
    N, T, m = 4096, 100, 8
    anc = synth.anchors_for(m)
    kw = dict(p_nlos=0.05, p_missing=0.02)
    with Batch(L.MODEL_T6, N, anchors=anc, accel_noise=0.5, ignore_worst_anchor=1) as b:
        one = synth.toa_montecarlo(b, T, T, anc, **kw)
        x1, P1, s1 = b.get_state()
        chunked = synth.toa_montecarlo(b, T, 25, anc, **kw)
        x2, P2, s2 = b.get_state()
    assert one.shape == (T, 6)
    assert np.array_equal(one, chunked)
    assert np.array_equal(x1, x2) and np.array_equal(P1, P2) and np.array_equal(s1, s2)
    s = epoch_summary(one)
    assert np.all(s["n"] == N) and np.all(np.isfinite(s["rmse"])) and s["rmse"][-1] < 0.5
    halves = []
    for ff in (0, N // 2):
        with Batch(L.MODEL_T6, N // 2, anchors=anc, accel_noise=0.5, ignore_worst_anchor=1) as b:
            rows = synth.toa_montecarlo(b, T, 40, anc, first_filter=ff, **kw)
            halves.append((rows, b.get_state()))
    assert np.array_equal(np.concatenate([h[1][0] for h in halves], axis=1), x1)
    assert np.array_equal(np.concatenate([h[1][1] for h in halves], axis=1), P1)
    assert np.array_equal(np.concatenate([h[1][2] for h in halves]), s1)
    # counts add up exactly; the sums to rounding (another summation tree)
    tot = halves[0][0] + halves[1][0]
    assert np.array_equal(tot[:, [2, 3, 5]], one[:, [2, 3, 5]])
    assert np.allclose(tot, one, rtol=1e-12, atol=0)


def test_toa_montecarlo_refuses_ml_batches():
    from roskfpos_b200.batch import Batch
    with Batch(L.MODEL_ML, 128, anchors=synth.anchors_for(8)) as b:
        with pytest.raises(ValueError):
            synth.toa_montecarlo(b, 10, 5, synth.anchors_for(8))


# --------------------------------------------------------------------------------------- 6. error paths
def test_error_paths():
    anc = np.ascontiguousarray(synth.anchors_for(8))
    t = np.arange(1, 5, dtype=np.float64) * 0.1
    import torch
    out = torch.empty((4, 8, 256), device=DEV, dtype=torch.int32)

    def call(n=256, M=8, T=4, fmt=L.FMT_I32_MM, a=anc, tt=t, o=out, g=None, **kw):
        g = g if g is not None else L.KfposSynthToa(**dict(dict(seed=1, tag_z=1.0, sigma_r=0.1, nlos_mean=0.8), **kw))
        return L.lib().kfpos_synth_toa_ranges(0, n, M, None if a is None else C.c_void_p(a.ctypes.data), T,
                                              None if tt is None else C.c_void_p(tt.ctypes.data),
                                              None if g is False else C.byref(g), fmt,
                                              None if o is None else C.c_void_p(o.data_ptr()), None)
    assert call() == 0
    bad = [dict(n=0), dict(n=-5), dict(M=0), dict(M=33), dict(T=-1), dict(a=None), dict(tt=None), dict(o=None),
           dict(g=False), dict(fmt=L.FMT_F64_M), dict(fmt=7), dict(p_missing=-0.1), dict(p_missing=1.5),
           dict(p_nlos=-0.01), dict(p_nlos=1.01), dict(p_missing=float("nan")), dict(sigma_r=-0.1),
           dict(sigma_r=float("nan")), dict(p_nlos=0.1, nlos_mean=0.0), dict(p_nlos=0.1, nlos_mean=-1.0),
           dict(first_filter=-1), dict(first_epoch=-1), dict(first_epoch=0xFFFFFFFF - 3),
           dict(first_epoch=0xFFFFFFFF)]
    for kw in bad:
        assert call(**kw) == -1, kw
    # edges that are valid: probabilities 0 and 1, no NLOS with any mean, the last epoch below the reserved index
    assert call(p_missing=1.0, p_nlos=1.0) == 0
    assert (out == 0).all()
    assert call(p_nlos=0.0, nlos_mean=0.0) == 0
    assert call(first_epoch=0xFFFFFFFF - 4) == 0
    assert call(T=0, tt=None, o=None) == 0
    with pytest.raises(L.KfposError):
        synth.toa_montecarlo_chunk(16, 0, 2, synth.anchors_for(8), DEV, p_missing=2.0)
    with pytest.raises(ValueError):
        synth.toa_montecarlo_chunk(16, 0, 2, synth.anchors_for(8), DEV, fmt=L.FMT_F64_M)
