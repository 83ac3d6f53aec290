"""Per-epoch Cramer-Rao bounds (kfpos_batch_crlb, Batch.crlb, synth.toa_montecarlo(crlb=...)): parity with a numpy
reference on generator logs and real selections, monotonicity, bit-exact sharding and chunking, the efficiency of
the ML estimator against its bound, the error paths and non-interference."""
import ctypes as C

import numpy as np
import pytest

from roskfpos_b200 import lib as L, synth

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
INVALID, NOT_READY, UNSUPPORTED = -1, -4, -5

# Anchor tables of the parity workloads (tag at z = 1).  Every set S that the workloads can produce with
# non-negligible probability has a Fisher information with a condition number below ~1e3 at every tag position of
# the Lissajous (checked on a grid of positions when the tables were chosen), so the FP64 sums of the kernel and of
# numpy, which round differently, agree to 1e-12 whatever the operation order.  The BASELINE tables do not have that
# property for small sets: 3 of the 4 config-1 anchors are coplanar with tag positions inside the room, and so are
# some 4-anchor groups of the 8-anchor table, where J becomes singular and its trace has no stable digits.
ANC4 = np.array([(-1, -1, 3.0), (11, -1, 2.6), (11, 11, 3.4), (-1, 11, 2.8)])
ANC8 = np.array([(x, y, z) for (x, y), z in zip([(0, 0), (5, 0), (10, 0), (10, 5), (10, 10), (5, 10), (0, 5), (0, 10)],
                                                [3.0, 5.0, 3.5, 4.5, 4.0, 3.2, 4.8, 3.7])])


def anchors(m):
    return {4: ANC4, 8: ANC8}[m] if m in (4, 8) else synth.anchors_for(m)


# ------------------------------------------------------------------------------------ numpy reference bound
def kept(ranges, sel=None, mode="none", nlos=None, set="present"):
    """The set S of kfpos_batch_crlb as a boolean [rows][M][N]: present (value > 0, NaN not; uint16 != 0), then
    minus the NLOS bits ("los") or minus what the selection dropped ("used": mode "none" keeps everything, "loo"
    drops the slot sel[r][f] when it is in [0, 32), "mask" keeps the bits of sel[r][f] read as uint32)."""
    r = np.asarray(ranges)
    r = r[None] if r.ndim == 2 else r
    R, M, N = r.shape
    S = (r != 0) if r.dtype == np.uint16 else (r > 0)
    a = np.arange(M, dtype=np.uint64)[None, :, None]
    if set == "los":
        nl = np.asarray(nlos).astype(np.int64).astype(np.uint64)[:R] & np.uint64(0xFFFFFFFF)
        S = S & (((nl[:, None, :] >> a) & np.uint64(1)) == 0)
    elif set == "used" and mode == "loo":
        s = np.asarray(sel, dtype=np.int64)[:R]
        S = S & (a.astype(np.int64) != s[:, None, :])
    elif set == "used" and mode == "mask":
        u = np.asarray(sel, dtype=np.int32)[:R].view(np.uint32).astype(np.uint64)
        S = S & (((u[:, None, :] >> a) & np.uint64(1)) == 1)
    return S


def reference_terms(truth, ranges, anc, var, dim=3, **kw):
    """The four terms of every (row, filter) of kfpos_batch_crlb, [rows][N][4], and the condition number of each
    J with a bound ([rows][N], NaN without).  truth [rows][3][N] (or [3][N]), ranges [rows][M][N] (or [M][N]), var a
    scalar or [rows][M][N]; kw: the set of `kept`."""
    tr = np.asarray(truth, dtype=np.float64)
    tr = tr[None] if tr.ndim == 2 else tr
    S = kept(ranges, **kw)
    R, M, N = S.shape
    v = np.broadcast_to(np.asarray(var, dtype=np.float64), (R, M, N)) if np.ndim(var) else np.full((R, M, N), var)
    v = v.reshape(R, M, N)
    A = np.asarray(anc, dtype=np.float64).reshape(-1, 3)[:M]
    with np.errstate(invalid="ignore", divide="ignore", over="ignore"):
        d = tr[:, None, :, :] - A[None, :, :, None]  # [R][M][3][N]
        g = d / np.sqrt((d * d).sum(axis=2))[:, :, None, :]
        w = np.where(S, 1.0 / v, 0.0)
        J = np.zeros((R, N, dim, dim))
        for i in range(dim):
            for j in range(dim):
                J[:, :, i, j] = np.where(S, w * g[:, :, i] * g[:, :, j], 0.0).sum(axis=1)
        ok = (S.sum(axis=1) >= dim) & np.isfinite(tr).all(axis=1) & np.where(S, (v > 0) & np.isfinite(v), True).all(axis=1)
        d0 = J[..., 0, 0]
        l10 = J[..., 1, 0] / d0
        d1 = J[..., 1, 1] - l10 * J[..., 1, 0]
        pd = (d0 > 0) & np.isfinite(d0) & (d1 > 0) & np.isfinite(d1)
        xx, yy, zz = 1 / d0 + l10 * l10 / d1, 1 / d1, 0.0
        if dim == 3:
            l20 = J[..., 2, 0] / d0
            c = J[..., 2, 1] - l20 * J[..., 1, 0]
            l21 = c / d1
            d2 = J[..., 2, 2] - l20 * J[..., 2, 0] - l21 * c
            pd &= (d2 > 0) & np.isfinite(d2)
            m20 = l20 - l10 * l21
            xx, yy, zz = xx + m20 * m20 / d2, yy + l21 * l21 / d2, 1 / d2
        xy = xx + yy
        trace = xy + zz
        ok &= pd & np.isfinite(trace)
        t = np.zeros((R, N, 4))
        t[..., 0] = np.where(ok, trace, 0.0)
        t[..., 1] = np.where(ok, xy, 0.0)
        t[..., 2] = ok
        t[..., 3] = ~ok
        Jf = np.where(ok[..., None, None], J, np.eye(dim))
        ev = np.linalg.eigvalsh(Jf)
        cond = np.where(ok, ev[..., -1] / ev[..., 0], np.nan)
    return t, cond


def reference_crlb(truth, ranges, anc, var, dim=3, **kw):
    """[rows][4] of kfpos_batch_crlb (sums in numpy's order; the kernel's tree agrees to rounding)."""
    return reference_terms(truth, ranges, anc, var, dim, **kw)[0].sum(axis=1)


def assert_parity(got, ref, cond, what):
    got, ref = np.asarray(got), np.asarray(ref)
    assert got.shape == ref.shape, (what, got.shape, ref.shape)
    assert np.array_equal(got[:, 2:], ref[:, 2:]), (what, got[:, 2:].sum(axis=0), ref[:, 2:].sum(axis=0))
    rel = np.abs(got[:, :2] - ref[:, :2]) / np.maximum(np.abs(ref[:, :2]), 1e-300)
    assert (rel[ref[:, :2] != 0] <= 1e-12).all() and (got[:, :2][ref[:, :2] == 0] == 0).all(), \
        (what, float(rel.max()), "largest condition number of J", float(np.nanmax(cond, initial=0)))


# --------------------------------------------------------------------------------------------- workloads
def chunk(n, T, m, epoch0=0, **kw):
    return synth.toa_montecarlo_chunk(n, epoch0, T, anchors(m), DEV, want_x0=True, want_truth=True, want_nlos=True,
                                      **kw)


def as_fmt(r_mm, fmt):
    """The int32 mm log in another wire format; f64 gets NaN for a third of its absent rangings (not present)."""
    if fmt == L.FMT_U16_MM:
        return np.ascontiguousarray(np.minimum(r_mm, 65535).astype(np.uint16))
    if fmt == L.FMT_F64_M:
        m = r_mm.astype(np.float64) / 1000.0
        m[(r_mm == 0) & (np.arange(r_mm.size).reshape(r_mm.shape) % 3 == 0)] = np.nan
        return m
    return r_mm


def per_ranging_var(shape, seed=7):
    """True variances that differ per ranging (0.005..0.03 m^2), so that the array path is not the scalar one."""
    return np.random.default_rng(seed).uniform(0.005, 0.03, size=shape)


def run_sets(b, truth, r, var, sel, nlos, device_args, sets=("present", "los", "used")):
    import torch
    out = {}
    for s in sets:
        if device_args:
            d = lambda a: None if a is None else (a if isinstance(a, float) else
                                                  torch.as_tensor(np.ascontiguousarray(a), device=DEV))
            o = torch.zeros((1 if b.model == L.MODEL_ML else r.shape[0], 4), dtype=torch.float64, device=DEV)
            b.crlb(d(truth), d(r), d(var), d(sel), d(nlos), set=s, out=o)
            out[s] = o.cpu().numpy()
        else:
            out[s] = b.crlb(truth, r, var, sel, nlos, set=s)
    return out


# ------------------------------------------------------------------------------------------ 1. parity, T6
T6_CASES = {
    "plain_m4": (4, {}, "none"),
    "plain_m8": (8, {}, "none"),
    "loo_m8": (8, dict(ignore_worst_anchor=1, ignore_cost_threshold=0.0), "loo"),
    "loo_m16": (16, dict(ignore_worst_anchor=1, ignore_cost_threshold=0.0), "loo"),
    "v1_m8": (8, dict(variant=1, num_ignored_rangings=1), "mask"),
    "v2_m8": (8, dict(variant=2, best_mode=0), "mask"),
    "v1_m32": (32, dict(variant=1, num_ignored_rangings=3), "mask"),
}


@pytest.mark.parametrize("fmt", [L.FMT_I32_MM, L.FMT_U16_MM, L.FMT_F64_M], ids=["i32", "u16", "f64"])
@pytest.mark.parametrize("case", list(T6_CASES))
def test_t6_parity(case, fmt):
    """Every set against numpy on a generator log with NLOS and missing rangings and the selection the T6 replay
    made on it; device pointers for int32, host arrays otherwise; a per-ranging variance for f64."""
    from roskfpos_b200.batch import Batch
    m, cfg, mode = T6_CASES[case]
    N, T = 4096, 8
    w = chunk(N, T, m, p_missing=0.01, p_nlos=0.02, nlos_mean=0.8)
    r = as_fmt(w["ranges"].cpu().numpy(), fmt)
    truth, nlos = w["truth"].cpu().numpy(), w["nlos"].cpu().numpy()
    var = per_ranging_var(r.shape) if fmt == L.FMT_F64_M else 0.01 + 1e-6 / 12
    with Batch(L.MODEL_T6, N, anchors=anchors(m), accel_noise=0.5, **cfg) as b:
        b.set_state(w["x0"].cpu().numpy())
        _, sel = b.replay_toa(0.1, r, err=0.10, want_sel=True)
        got = run_sets(b, truth, r, var, sel if mode != "none" else None, nlos, fmt == L.FMT_I32_MM)
    for s, g in got.items():
        ref, cond = reference_terms(truth, r, anchors(m), var, 3, sel=sel, mode=mode, nlos=nlos, set=s)
        assert_parity(g, ref.sum(axis=1), cond, (case, s))
        assert g[:, 2].sum() > 0


@pytest.mark.parametrize("N", [1000, 129])
def test_t6_parity_ragged_batches(N):
    """Batches that end inside a warp (lanes without a filter add zeros) and inside a block."""
    from roskfpos_b200.batch import Batch
    m, cfg, mode = T6_CASES["v1_m8"]
    w = chunk(N, 6, m, p_missing=0.01, p_nlos=0.02)
    r, truth, nlos = w["ranges"].cpu().numpy(), w["truth"].cpu().numpy(), w["nlos"].cpu().numpy()
    with Batch(L.MODEL_T6, N, anchors=anchors(m), accel_noise=0.5, **cfg) as b:
        b.set_state(w["x0"].cpu().numpy())
        _, sel = b.replay_toa(0.1, r, err=0.10, want_sel=True)
        got = run_sets(b, truth, r, 0.01, sel, nlos, N == 129)
    for s, g in got.items():
        ref, cond = reference_terms(truth, r, anchors(m), 0.01, 3, sel=sel, mode=mode, nlos=nlos, set=s)
        assert_parity(g, ref.sum(axis=1), cond, (N, s))


# ------------------------------------------------------------------------------------- 1. parity, K8 and T9
@pytest.mark.parametrize("m", [4, 8])
@pytest.mark.parametrize("model", [L.MODEL_K8, L.MODEL_T9], ids=["k8", "t9"])
def test_k8_t9_parity(model, m):
    """PRESENT and LOS need no selection: K8 bounds the x-y position (D = 2, over the 3-D distance), T9 all three
    coordinates.  A K8 log at 4 anchors has no impairments: two rangings leave the 2-D J singular on lines that
    cross the room."""
    from roskfpos_b200.batch import Batch
    N, T = 4096, 8
    dim = 2 if model == L.MODEL_K8 else 3
    w = chunk(N, T, m, **(dict(p_missing=0.01, p_nlos=0.02) if dim == 3 or m == 8 else {}))
    r, truth, nlos = w["ranges"].cpu().numpy(), w["truth"].cpu().numpy(), w["nlos"].cpu().numpy()
    var = per_ranging_var(r.shape, seed=m)
    with Batch(model, N, anchors=anchors(m)) as b:
        got = run_sets(b, truth, r, var, None, nlos, m == 8, sets=("present", "los"))
    for s, g in got.items():
        ref, cond = reference_terms(truth, r, anchors(m), var, dim, nlos=nlos, set=s)
        assert_parity(g, ref.sum(axis=1), cond, (model, m, s))
        assert g[:, 2].sum() > 0
    if dim == 2:
        assert np.array_equal(got["present"][:, 0], got["present"][:, 1])  # tr J^-1 is the x-y part


# ------------------------------------------------------------------------------------------ 1. parity, ML
ML_CASES = {
    "v0": (8, dict(variant=0), "none", 3),
    "v0_m4": (4, dict(variant=0), "none", 3),
    "v1": (8, dict(variant=1, num_ignored_rangings=1), "mask", 3),
    "v2": (8, dict(variant=2, best_mode=0), "mask", 3),
    "v0_2d": (8, dict(variant=0, use2d=1), "none", 2),
    "v2_2d": (8, dict(variant=2, use2d=1), "mask", 2),
}


@pytest.mark.parametrize("fmt", [L.FMT_I32_MM, L.FMT_F64_M], ids=["i32", "f64"])
@pytest.mark.parametrize("case", list(ML_CASES))
def test_ml_parity(case, fmt):
    """One epoch per ML batch: truth [3][N], log [M][N], the final selection in row 0 of sel [2][N]."""
    from roskfpos_b200.batch import Batch
    m, cfg, mode, dim = ML_CASES[case]
    N = 4096
    w = chunk(N, 1, m, epoch0=3, p_missing=0.01, p_nlos=0.05)
    r = as_fmt(w["ranges"].cpu().numpy()[0], fmt)
    truth, nlos = w["truth"].cpu().numpy()[0], w["nlos"].cpu().numpy()
    var = per_ranging_var(r.shape) if fmt == L.FMT_F64_M else 0.01
    with Batch(L.MODEL_ML, N, anchors=anchors(m), **cfg) as b:
        out = b.ml_solve(r, err=0.10)
        got = run_sets(b, truth, r, var, out["sel"] if mode != "none" else None, nlos, fmt == L.FMT_I32_MM)
    for s, g in got.items():
        ref, cond = reference_terms(truth, r, anchors(m), var, dim, sel=out["sel"], mode=mode, nlos=nlos, set=s)
        assert_parity(g, ref.sum(axis=1), cond, (case, s))
        assert g[0, 2] > 0
    if mode == "mask":
        assert got["used"][0, 0] > got["present"][0, 0]


def test_used_mask_with_32_anchors():
    """A full 32-anchor mask is -1 (bit 31 is the sign bit) and drops nothing; 0x7fffffff drops slot 31."""
    from roskfpos_b200.batch import Batch
    N = 2048
    w = chunk(N, 2, 32)
    r, truth = w["ranges"].cpu().numpy(), w["truth"].cpu().numpy()
    sel = np.full((2, N), -1, dtype=np.int32)
    sel[:, 1::2] = 0x7FFFFFFF
    with Batch(L.MODEL_T6, N, anchors=anchors(32), accel_noise=0.5, variant=1, num_ignored_rangings=1) as b:
        got = b.crlb(truth, r, 0.01, sel, set="used")
        full = b.crlb(truth, r, 0.01, np.full((2, N), -1, dtype=np.int32), set="used")
        pres = b.crlb(truth, r, 0.01, set="present")
    ref, cond = reference_terms(truth, r, anchors(32), 0.01, 3, sel=sel, mode="mask", set="used")
    assert_parity(got, ref.sum(axis=1), cond, "m32")
    assert np.array_equal(full, pres) and (got[:, 0] > pres[:, 0]).all()


# ------------------------------------------------------------------------------------------ 2. monotonicity
def test_fewer_rangings_never_lower_the_bound():
    """Removing rangings can only raise tr J^-1 (J loses a positive semi-definite term).  At 3 % NLOS no filter is
    left with fewer than 3 LOS rangings of 8 (expected 0.003 times in the run; at 10 % it happened 3 times), so
    every filter keeps its bound in every set and the row sums compare filter by filter."""
    from roskfpos_b200.batch import Batch, crlb_summary
    N, T, m = 4096, 30, 8
    with Batch(L.MODEL_T6, N, anchors=anchors(m), accel_noise=0.5, variant=1, num_ignored_rangings=1) as b:
        rows, cr = synth.toa_montecarlo(b, T, T, anchors(m), p_nlos=0.03, crlb=("present", "los", "used"))
    for s in cr:
        assert (cr[s][:, 2] == N).all() and not cr[s][:, 3].any(), s  # every filter has a bound
    assert (cr["los"][:, 0] >= cr["present"][:, 0]).all() and (cr["used"][:, 0] >= cr["present"][:, 0]).all()
    assert (cr["los"][:, 1] >= cr["present"][:, 1]).all() and (cr["used"][:, 1] >= cr["present"][:, 1]).all()
    assert (cr["used"][:, 0] > cr["present"][:, 0]).all()  # variant 1 drops a ranging in every epoch
    s = crlb_summary(cr["present"])
    assert (s["rmse_bound"] > 0.03).all() and (s["rmse_bound"] < 0.5).all() and (s["n"] == N).all()


# ------------------------------------------------------------------------------ 3. sharding and chunking
def test_aligned_shards_and_row_chunks_are_bit_exact():
    import torch
    from roskfpos_b200.batch import Batch, rank_tree
    N, T, m = 4096, 12, 8
    anc = anchors(m)
    w = chunk(N, T, m, p_missing=0.02, p_nlos=0.05)
    with Batch(L.MODEL_T6, N, anchors=anc, accel_noise=0.5, variant=1, num_ignored_rangings=1) as b:
        b.set_state(w["x0"])
        sel = torch.empty((T, N), dtype=torch.int32, device=DEV)
        b.replay_toa(0.1, w["ranges"], err=0.10, sel=sel)
        whole = {s: b.crlb(w["truth"], w["ranges"], 0.01, sel, w["nlos"], set=s) for s in ("present", "los", "used")}
    for G in (2, 4):
        n = N // G
        for s in whole:
            ranks = []
            for k in range(G):
                cut = lambda a: a[..., k * n:(k + 1) * n].contiguous()
                with Batch(L.MODEL_T6, n, anchors=anc, accel_noise=0.5, variant=1, num_ignored_rangings=1) as b:
                    ranks.append(b.crlb(cut(w["truth"]), cut(w["ranges"]), 0.01, cut(sel), cut(w["nlos"]), set=s))
            assert np.array_equal(rank_tree(ranks), whole[s]), (G, s)


def test_one_call_equals_row_chunks():
    """1000 rows in one call equal four calls of 250; and 260 rows of 1 Mi filters (two batches of the 256 MB
    partials scratch: 256 + 4 rows) equal calls of 100 rows (one batch each)."""
    from roskfpos_b200.batch import Batch
    for N, T, step in ((1024, 1000, 250), (1 << 20, 260, 100)):
        w = chunk(N, T, 8, p_missing=0.02, p_nlos=0.05)
        with Batch(L.MODEL_T6, N, anchors=anchors(8), accel_noise=0.5) as b:
            one = b.crlb(w["truth"], w["ranges"], 0.01, None, w["nlos"], set="los")
            parts = np.concatenate([b.crlb(w["truth"][k:k + step], w["ranges"][k:k + step], 0.01, None,
                                           w["nlos"][k:k + step], set="los") for k in range(0, T, step)])
        assert one.shape == (T, 4) and np.array_equal(one, parts), N
        del w


def test_montecarlo_whole_and_chunked():
    from roskfpos_b200.batch import Batch
    N, T, m = 4096, 60, 8
    sets = ("present", "los", "used")
    kw = dict(p_nlos=0.05, p_missing=0.02, sigma_r=0.1)
    with Batch(L.MODEL_T6, N, anchors=anchors(m), accel_noise=0.5, variant=2) as b:
        rows, sc, cr = synth.toa_montecarlo(b, T, T, anchors(m), score=True, crlb=sets, **kw)
        rows_c, cr_c = synth.toa_montecarlo(b, T, 25, anchors(m), crlb=sets, **kw)
        rows_p = synth.toa_montecarlo(b, T, 25, anchors(m), **kw)
    assert set(cr) == set(sets) and all(cr[s].shape == (T, 4) for s in sets)
    for s in sets:
        assert np.array_equal(cr[s], cr_c[s]), s
    assert np.array_equal(rows, rows_c) and np.array_equal(rows, rows_p)  # the bound changes no statistic
    assert sc.shape == (T, 8)


# --------------------------------------------------------------------------------------- 4. efficiency
@pytest.mark.parametrize("use2d", [False, True], ids=["3d", "2d"])
def test_ml_is_efficient_without_impairments(use2d):
    """At sigma_r 0.10 m with 8 anchors and no NLOS, the snapshot ML estimator is nearly efficient: its MSE over
    64 Ki epochs is the mean PRESENT floor to within a few per cent."""
    import torch
    from roskfpos_b200.batch import Batch
    N, m, tag_z = 1 << 16, 8, 1.0
    anc = synth.anchors_for(m)
    w = synth.toa_montecarlo_chunk(N, 0, 1, anc, DEV, sigma_r=0.10, tag_z=tag_z, want_truth=True)
    cfg = dict(variant=0, use2d=1, ml_start=(5.0, 5.0, tag_z)) if use2d else dict(variant=0, ml_start=(5.0, 5.0, 1.5))
    with Batch(L.MODEL_ML, N, anchors=anc, **cfg) as b:
        out = b.ml_solve(w["ranges"][0], err=0.10)
        bound = b.crlb(w["truth"][0], w["ranges"][0], 0.10 ** 2 + 1e-6 / 12)
    truth = w["truth"][0].cpu().numpy()
    e = out["pos"] - truth
    e2 = (e[:2] ** 2).sum(axis=0) if use2d else (e ** 2).sum(axis=0)
    ok = (out["status"] == 0) & np.isfinite(e2)
    assert ok.mean() > 0.999
    assert bound[0, 2] == N and bound[0, 3] == 0
    ratio = e2[ok].mean() / (bound[0, 0] / bound[0, 2])
    print("ML MSE / CRLB", "2d" if use2d else "3d", ratio)
    assert 0.95 <= ratio <= 1.10, ratio
    torch.cuda.synchronize()


# ------------------------------------------------------------------------------------ 5. errors, state
def test_error_paths():
    from roskfpos_b200.batch import Batch
    lib = L.lib()
    N, T, M = 256, 3, 8
    anc = anchors(M)
    truth = np.full((T, 3, N), 5.0)
    r = np.full((T, M, N), 5000, dtype=np.int32)
    sel = np.full((T, N), -1, dtype=np.int32)
    nlos = np.zeros((T, N), dtype=np.uint32)
    var = np.full((T, M, N), 0.01)
    out = np.zeros((T, 4))
    hp = lambda a: None if a is None else C.c_void_p(a.ctypes.data)

    def call(b, s=L.CRLB_PRESENT, rows=T, tr=truth, ranges=r, fmt=L.FMT_I32_MM, vs=0.01, v=None, sl=sel, nl=nlos,
             o=out):
        return lib.kfpos_batch_crlb(b, s, rows, hp(tr), hp(ranges), fmt, vs, hp(v), hp(sl), hp(nl), hp(o), None)
    assert call(None) == INVALID
    with Batch(L.MODEL_T6, N, accel_noise=0.5, ignore_worst_anchor=1) as b:
        assert call(b._h) == NOT_READY
        b.set_anchors(anc)
        for s in (L.CRLB_PRESENT, L.CRLB_LOS, L.CRLB_USED):
            assert call(b._h, s=s) == 0
        assert call(b._h, vs=float("nan"), v=var) == 0  # the scalar is not read with an array
        for kw in (dict(s=3), dict(s=-1), dict(rows=0), dict(rows=-1), dict(fmt=3), dict(fmt=-1), dict(tr=None),
                   dict(ranges=None), dict(o=None), dict(vs=0.0), dict(vs=-1.0), dict(vs=float("nan")),
                   dict(vs=float("inf")), dict(s=L.CRLB_LOS, nl=None), dict(s=L.CRLB_USED, sl=None)):
            assert call(b._h, **kw) == INVALID, kw
        assert call(b._h, s=L.CRLB_PRESENT, sl=None, nl=None) == 0
    with Batch(L.MODEL_T6, N, anchors=anc, accel_noise=0.5) as b:
        assert call(b._h, s=L.CRLB_USED, sl=None) == 0  # plain T6 drops nothing: sel is not read
    for cfg in (dict(variant=1), dict(variant=2)):
        with Batch(L.MODEL_T6, N, anchors=anc, accel_noise=0.5, **cfg) as b:
            assert call(b._h, s=L.CRLB_USED, sl=None) == INVALID
    for model in (L.MODEL_K8, L.MODEL_T9):
        with Batch(model, N, anchors=anc) as b:
            assert call(b._h, s=L.CRLB_USED) == UNSUPPORTED
            assert call(b._h, s=L.CRLB_PRESENT) == 0 and call(b._h, s=L.CRLB_LOS) == 0
    with Batch(L.MODEL_ML, N, anchors=anc, variant=1, num_ignored_rangings=1) as b:
        ml_sel = np.full((2, N), -1, dtype=np.int32)
        assert call(b._h, s=L.CRLB_USED, rows=1, tr=truth[0], ranges=r[0], sl=ml_sel) == 0
        assert call(b._h, rows=2) == INVALID
        assert call(b._h, s=L.CRLB_USED, rows=1, tr=truth[0], ranges=r[0], sl=None) == INVALID
    with Batch(L.MODEL_ML, N, anchors=anc) as b:
        assert call(b._h, s=L.CRLB_USED, rows=1, tr=truth[0], ranges=r[0], sl=None) == 0  # variant 0


def test_bound_leaves_the_batch_untouched():
    from roskfpos_b200.batch import Batch
    N, T, m = 2048, 10, 8
    w = chunk(N, T, m, p_nlos=0.05)
    with Batch(L.MODEL_T6, N, anchors=anchors(m), accel_noise=0.5, ignore_worst_anchor=1) as b:
        b.set_state(w["x0"])
        _, sel = b.replay_toa(0.1, w["ranges"], err=0.1, want_sel=True)
        before = b.get_state(), b.counters()
        for s in ("present", "los", "used"):
            b.crlb(w["truth"], w["ranges"], 0.01, sel, w["nlos"], set=s)
        after = b.get_state(), b.counters()
    for a, c in zip(before[0], after[0]):
        assert np.array_equal(a, c)
    assert before[1] == after[1]
