"""Obstacle-based NLOS of the ranging generator (kfpos_synth_toa_ranges_geo, DESIGN §4.5f): the slab decision
of every ranging reproduced bit for bit by numpy from the device truth, the documented excess, exponential bias
and loss draws, identity with the plain generator where no box blocks, purity under sharding and chunking, and
the Monte Carlo bench on top of it."""
import ctypes as C

import numpy as np
import pytest

from roskfpos_b200 import lib as L, synth
from tests.test_gpu_synth_toa import M32, distances_mm, impairment_uniforms, philox, uniform2

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
# the study scenario of DESIGN §4.5f: pillar, partition, metal cabinet
STUDY = np.array([[1.2, 7.6, 0.0, 1.8, 8.2, 3.0, 1.2, 0.2, 0.1],
                  [8.6, 2.0, 0.0, 8.75, 3.5, 2.2, 0.6, 0.1, 0.05],
                  [3.6, 8.4, 0.0, 4.6, 8.9, 1.2, 0.0, 1.0, 0.5]])
# above the 2.5 m anchors: blocks nothing
CEILING = np.array([[0.0, 0.0, 3.0, 10.0, 10.0, 3.5, 1.0, 1.0, 0.5],
                    [4.0, 4.0, 2.6, 6.0, 6.0, 2.7, 2.0, 0.5, 1.0]])


def table(rows):
    rows = np.asarray(rows, dtype=np.float64).reshape(-1, 9)
    tbl = (L.KfposObstacle * max(len(rows), 1))()
    for o, b in zip(tbl, rows):
        o.lo[:], o.hi[:] = b[0:3], b[3:6]
        o.excess_per_m, o.spread, o.p_loss = b[6], b[7], b[8]
    return tbl


def geo(n, epoch0, T, boxes, anc=None, fmt=L.FMT_I32_MM, mask=True, first_filter=0, seed=synth.SEED, **kw):
    """kfpos_synth_toa_ranges_geo through the C ABI into device buffers: host (ranges, nlos or None)."""
    import torch
    anc = np.ascontiguousarray(synth.anchors_for(8) if anc is None else anc, dtype=np.float64)
    M = len(anc)
    t = np.ascontiguousarray(np.arange(epoch0 + 1, epoch0 + T + 1, dtype=np.float64) * 0.1)
    r = torch.empty((T, M, n), dtype=torch.uint16 if fmt == L.FMT_U16_MM else torch.int32, device=DEV)
    m = torch.empty((T, n), dtype=torch.int32, device=DEV) if mask else None
    g = L.KfposSynthToa(**dict(dict(seed=seed, first_filter=first_filter, first_epoch=epoch0, tag_z=1.0,
                                    sigma_r=0.1, nlos_mean=0.8), **kw))
    boxes = np.asarray(boxes, dtype=np.float64).reshape(-1, 9)
    L.check(L.lib().kfpos_synth_toa_ranges_geo(0, n, M, C.c_void_p(anc.ctypes.data), T, C.c_void_p(t.ctypes.data),
                                               C.byref(g), len(boxes), C.cast(table(boxes), C.c_void_p), fmt,
                                               C.c_void_p(r.data_ptr()), None if m is None else C.c_void_p(m.data_ptr()),
                                               None), "kfpos_synth_toa_ranges_geo")
    return r.cpu().numpy(), None if m is None else m.cpu().numpy().view(np.uint32)


def plain(n, epoch0, T, anc=None, fmt=L.FMT_I32_MM, **kw):
    """The same arguments through kfpos_synth_toa_ranges_nlos (synth.toa_montecarlo_chunk): ranges, mask, truth."""
    kw = dict(dict(sigma_r=0.1), **kw)
    w = synth.toa_montecarlo_chunk(n, epoch0, T, synth.anchors_for(8) if anc is None else anc, DEV, fmt=fmt,
                                   want_nlos=True, want_truth=True, **kw)
    return w["ranges"].cpu().numpy(), w["nlos"].cpu().numpy().view(np.uint32), w["truth"].cpu().numpy()


def slab(truth, anc, boxes):
    """numpy slab test of DESIGN §4.5f on the device truth [T][3][N]: per box blocked [T][M][N] and the fraction
    (exit - enter) of the segment inside it, with the same single IEEE operations as the kernel."""
    tp = truth[:, None, :, :]                   # [T][1][3][N]
    dv = anc[None, :, :, None] - tp             # [T][M][3][N]
    with np.errstate(divide="ignore"):
        inv = 1.0 / dv
    out = []
    for b in np.asarray(boxes, dtype=np.float64).reshape(-1, 9):
        enter = np.zeros(dv[:, :, 0].shape)
        exit_ = np.ones(dv[:, :, 0].shape)
        inside = np.ones(dv[:, :, 0].shape, dtype=bool)
        for j in range(3):
            nz = dv[:, :, j] != 0.0
            with np.errstate(invalid="ignore"):
                s1 = (b[j] - tp[:, :, j]) * inv[:, :, j]
                s2 = (b[3 + j] - tp[:, :, j]) * inv[:, :, j]
            enter = np.where(nz, np.fmax(enter, np.fmin(s1, s2)), enter)
            exit_ = np.where(nz, np.fmin(exit_, np.fmax(s1, s2)), exit_)
            inside &= nz | ((b[j] < tp[:, :, j]) & (tp[:, :, j] < b[3 + j]))
        blk = inside & (enter < exit_)
        out.append((blk, np.where(blk, exit_ - enter, 0.0)))
    return out


def geo_uniforms(seed, first_filter, N, epoch0, T, M):
    """(u, v) [T][M][N] of the counters (gf lo, gf hi, g, 0x40000000 | a)."""
    gf = np.uint64(first_filter) + np.arange(N, dtype=np.uint64)
    g = (np.uint64(epoch0) + np.arange(T, dtype=np.uint64))[:, None, None]
    a = (np.uint64(0x40000000) | np.arange(M, dtype=np.uint64))[None, :, None]
    c = philox((gf & M32)[None, None, :], (gf >> np.uint64(32))[None, None, :], g, a, seed & 0xFFFFFFFF, seed >> 32)
    return uniform2([np.broadcast_to(v, (T, M, N)) for v in c])


def model(truth, anc, boxes):
    """blocked, sum excess * L (m), sum spread, 1 - prod(1 - p_loss): [T][M][N] from the numpy slab test."""
    d = distances_mm(truth, anc) / 1000.0
    blocked = np.zeros(d.shape, dtype=bool)
    excess, spread, keep = np.zeros(d.shape), np.zeros(d.shape), np.ones(d.shape)
    for b, (blk, frac) in zip(np.asarray(boxes, dtype=np.float64).reshape(-1, 9), slab(truth, anc, boxes)):
        blocked |= blk
        excess += np.where(blk, b[6] * frac * d, 0.0)
        spread += np.where(blk, b[7], 0.0)
        keep = np.where(blk, keep * (1.0 - b[8]), keep)
    return blocked, excess, spread, 1.0 - keep


def bits(mask_tmn):
    """[T][M][N] bool -> [T][N] uint32 with bit a of anchor a."""
    w = (np.uint32(1) << np.arange(mask_tmn.shape[1], dtype=np.uint32))[None, :, None]
    return (mask_tmn.astype(np.uint32) * w).sum(axis=1, dtype=np.uint64).astype(np.uint32)


def hand_anchors():
    """anchors_for(8) plus two at the tag height (segments parallel to the floor: Dv_z == 0)."""
    return np.ascontiguousarray(np.vstack([synth.anchors_for(8), [[5.0, 5.0, 1.0], [9.5, 1.0, 1.0]]]))


HAND = np.array([[4.9, -1.0, 0.0, 5.1, 11.0, 2.0, 0.5, 0.0, 0.0],   # a wall at x = 5 across the room, z (0, 2)
                 [0.0, 0.0, 0.0, 10.0, 10.0, 1.5, 0.3, 0.0, 0.0],   # the tag's whole range inside a box
                 [2.0, 2.0, 0.2, 8.0, 8.0, 1.0, 0.7, 0.0, 0.0],     # top face at the tag height: grazed by Dv_z == 0
                 [2.0, 2.0, 1.0, 8.0, 8.0, 1.8, 0.9, 0.0, 0.0]])    # bottom face at the tag height


# ------------------------------------------------------------------------------------------------ 1. identity
@pytest.mark.parametrize("fmt", [L.FMT_I32_MM, L.FMT_U16_MM])
@pytest.mark.parametrize("impair", [False, True])
def test_no_boxes_or_boxes_that_block_nothing_change_no_byte(fmt, impair):
    N, T = 3000, 40
    kw = dict(p_missing=0.1, p_nlos=0.1) if impair else {}
    r0, m0, _ = plain(N, 5, T, fmt=fmt, **kw)
    for boxes in (np.zeros((0, 9)), CEILING):
        r, m = geo(N, 5, T, boxes, fmt=fmt, **kw)
        assert np.array_equal(r, r0) and np.array_equal(m, m0)
        r, none = geo(N, 5, T, boxes, fmt=fmt, mask=False, **kw)
        assert none is None and np.array_equal(r, r0)
    w = synth.toa_montecarlo_chunk(N, 5, T, synth.anchors_for(8), DEV, fmt=fmt, obstacles=CEILING, **kw)
    assert np.array_equal(w["ranges"].cpu().numpy(), r0)


# ------------------------------------------------------------------------------------------------ 2. decision
@pytest.mark.parametrize("case", ["study", "hand"])
def test_mask_equals_numpy_slab_test(case):
    """sigma_r = 0, no i.i.d. impairments, p_loss = 0: the mask is the numpy slab test, bit for bit.  The hand-made
    boxes go one per call, so that the box holding the tag's whole range does not hide the others."""
    N, T, epoch0 = 4096, 50, 17
    anc, boxes = (synth.anchors_for(8), STUDY) if case == "study" else (hand_anchors(), HAND)
    boxes = boxes.copy()
    boxes[:, 8] = 0.0
    _, _, truth = plain(N, epoch0, T, anc=anc)
    for bx in ([boxes] if case == "study" else [boxes[i:i + 1] for i in range(len(boxes))]):
        r, m = geo(N, epoch0, T, bx, anc=anc, sigma_r=0.0)
        blocked = model(truth, anc, bx)[0]
        assert (r > 0).all()
        assert np.array_equal(m, bits(blocked))
    if case == "study":
        assert 0.01 < blocked.mean() < 0.5
    else:
        blk = [b for b, _ in slab(truth, anc, boxes)]
        # the wall at x = 5 blocks the z-level anchor 9 at (9.5, 1) from the tags west of it only
        assert blk[0][:, 9].any() and not blk[0][:, 9].all()
        # tag inside box 1: every segment starts inside it, so the box blocks every ranging
        assert blk[1].all()
        # the z-level anchors 8 and 9 run in the plane of a face of boxes 2 and 3: open boxes do not block them
        assert not blk[2][:, 8:].any() and not blk[3][:, 8:].any()
        # the other anchors' segments cross those boxes
        assert blk[2][:, :8].any() and blk[3][:, :8].any()


# ---------------------------------------------------------------------------------------------------- 3. bias
@pytest.mark.parametrize("case", ["study", "hand"])
def test_excess_and_exponential_bias(case):
    N, T, epoch0, seed = 4096, 30, 3, 77
    anc, boxes = (synth.anchors_for(8), STUDY) if case == "study" else (hand_anchors(), HAND)
    boxes = boxes.copy()
    boxes[:, 8] = 0.0
    _, _, truth = plain(N, epoch0, T, anc=anc, seed=seed)
    d = distances_mm(truth, anc)
    blocked, excess, spread, _ = model(truth, anc, boxes)
    no_spread = boxes.copy()
    no_spread[:, 7] = 0.0
    r, _ = geo(N, epoch0, T, no_spread, anc=anc, sigma_r=0.0, seed=seed)
    assert np.abs(r - np.floor(d + excess * 1000.0)).max() <= 1
    assert (excess[blocked] > 0).any() if case == "study" else (excess[blocked] > 0).all()
    r, _ = geo(N, epoch0, T, boxes, anc=anc, sigma_r=0.0, seed=seed)
    _, v = geo_uniforms(seed, 0, N, epoch0, T, len(anc))
    bias = np.where(blocked & (spread > 0), -spread * np.log(v), 0.0)
    assert np.abs(r - np.floor(d + (excess + bias) * 1000.0)).max() <= 1
    if case == "study":
        assert (bias > 0).any()


# ---------------------------------------------------------------------------------------------------- 4. loss
def test_loss_draws():
    N, T, epoch0, seed, ff = 4096, 40, 1000, 0x1234567890ABCDEF, 123456789
    anc = synth.anchors_for(8)
    boxes = STUDY.copy()
    boxes[2, 8] = 0.6
    _, _, truth = plain(N, epoch0, T, seed=seed, first_filter=ff)
    blocked, _, _, p_lost = model(truth, anc, boxes)
    u, _ = geo_uniforms(seed, ff, N, epoch0, T, 8)
    r, m = geo(N, epoch0, T, boxes, sigma_r=0.0, seed=seed, first_filter=ff)
    lost = blocked & (u < p_lost)
    assert np.array_equal(r == 0, lost)
    assert lost.any() and not lost.all()
    assert (r[~blocked] > 0).all()  # an unblocked ranging is never lost to geometry
    assert np.array_equal(m, bits(blocked & ~lost))
    # p_loss = 1: every blocked ranging is absent, and the mask is empty
    boxes[:, 8] = 1.0
    r, m = geo(N, epoch0, T, boxes, sigma_r=0.0, seed=seed, first_filter=ff)
    assert np.array_equal(r == 0, blocked) and not m.any()


# ------------------------------------------------------------------------------- 5. with i.i.d. impairments
@pytest.mark.parametrize("fmt", [L.FMT_I32_MM, L.FMT_U16_MM])
def test_combination_with_iid_impairments(fmt):
    N, T, epoch0, seed = 4096, 40, 9, 5
    anc = synth.anchors_for(8)
    kw = dict(p_missing=0.1, p_nlos=0.1, nlos_mean=0.8, seed=seed)
    r0, m0, truth = plain(N, epoch0, T, fmt=fmt, **kw)
    r, m = geo(N, epoch0, T, STUDY, fmt=fmt, **kw)
    blocked = model(truth, anc, STUDY)[0]
    u, v = impairment_uniforms(seed, 0, N, epoch0, T, 8)
    # the unblocked rangings are the plain generator's, byte for byte; the i.i.d.-missing ones stay absent
    assert np.array_equal(r[~blocked], r0[~blocked])
    assert (r[u < 0.1] == 0).all()
    present = r > 0
    assert np.array_equal(m, bits((blocked | (v < 0.1)) & present))
    assert not np.array_equal(m, m0)


# --------------------------------------------------------------------------------------------------- 6. purity
def test_shards_chunks_and_long_calls_are_bit_exact():
    kw = dict(p_missing=0.05, p_nlos=0.05)
    N, T = 2048, 2100  # more than the 1024 epochs of one launch
    r, m = geo(N, 0, T, STUDY, **kw)
    rs, ms = geo(500, 0, T, STUDY, first_filter=1000, **kw)
    assert np.array_equal(rs, r[:, :, 1000:1500]) and np.array_equal(ms, m[:, 1000:1500])
    rc, mc = geo(N, 1500, 600, STUDY, **kw)
    assert np.array_equal(rc, r[1500:]) and np.array_equal(mc, m[1500:])
    w = synth.toa_montecarlo_chunk(N, 1500, 600, synth.anchors_for(8), DEV, obstacles=STUDY, want_nlos=True, **kw)
    assert np.array_equal(w["ranges"].cpu().numpy(), rc)
    assert np.array_equal(w["nlos"].cpu().numpy().view(np.uint32), mc)


# ---------------------------------------------------------------------------------------------- 7. the bench
def test_toa_montecarlo_with_obstacles():
    from roskfpos_b200.batch import Batch, crlb_summary
    N, T = 4096, 60
    anc = synth.anchors_for(8)
    sets = ("present", "los", "used")
    out = []
    for chunk in (T, 25):
        with Batch(L.MODEL_T6, N, anchors=anc, accel_noise=0.5, variant=1, num_ignored_rangings=1) as b:
            out.append(synth.toa_montecarlo(b, T, chunk, anc, err=0.10, score=True, crlb=sets, obstacles=STUDY))
    (rows, sc, cr), (rows2, sc2, cr2) = out
    assert np.array_equal(rows, rows2) and np.array_equal(sc, sc2)
    for s in sets:
        assert np.array_equal(cr[s], cr2[s])
    # the scorer counted the NLOS rangings of the geometric mask
    w = synth.toa_montecarlo_chunk(N, 0, T, anc, DEV, obstacles=STUDY, want_nlos=True)
    nl = w["nlos"].cpu().numpy().view(np.uint8).reshape(T, -1)
    assert np.array_equal(sc[:, 2], np.unpackbits(nl, axis=1).sum(axis=1))
    assert sc[:, 2].min() > 0
    p, los = crlb_summary(cr["present"]), crlb_summary(cr["los"])
    assert np.array_equal(p["n"], los["n"])
    assert (los["rmse_bound"] >= p["rmse_bound"]).all()
    assert (los["rmse_bound"] > p["rmse_bound"]).any()


# ---------------------------------------------------------------------------------- 8. errors and the sync rule
def test_error_paths():
    import torch
    anc = np.ascontiguousarray(synth.anchors_for(8))
    t = np.arange(1, 5, dtype=np.float64) * 0.1
    out = torch.zeros((4, 8, 256), device=DEV, dtype=torch.int32)
    good = list(STUDY[0])

    def call(rows=(good,), n=None, tbl=True, M=8, fmt=L.FMT_I32_MM, **kw):
        g = L.KfposSynthToa(**dict(dict(seed=1, tag_z=1.0, sigma_r=0.1, nlos_mean=0.8), **kw))
        n = len(rows) if n is None else n
        return L.lib().kfpos_synth_toa_ranges_geo(0, 256, M, C.c_void_p(anc.ctypes.data), 4, C.c_void_p(t.ctypes.data),
                                                  C.byref(g), n, C.cast(table(rows), C.c_void_p) if tbl else None, fmt,
                                                  C.c_void_p(out.data_ptr()), None, None)
    assert call() == 0
    assert call(rows=(), tbl=False) == 0
    assert call(rows=[good] * L.MAX_OBSTACLES) == 0
    # what kfpos_synth_toa_ranges refuses
    for kw in (dict(M=0), dict(M=33), dict(fmt=L.FMT_F64_M), dict(p_missing=1.5), dict(sigma_r=-0.1),
               dict(p_nlos=0.1, nlos_mean=0.0), dict(first_filter=-1), dict(first_epoch=0xFFFFFFFF)):
        assert call(**kw) == -1, kw
    assert call(n=-1) == -1
    assert call(rows=[good] * (L.MAX_OBSTACLES + 1)) == -1
    assert call(n=1, tbl=False) == -1
    nan, inf = float("nan"), float("inf")
    for j, v in [(j, v) for j in range(6) for v in (nan, inf, -inf)] + [(6, -0.5), (6, nan), (6, inf), (7, -0.5),
                                                                        (7, nan), (7, inf), (8, -0.1), (8, 1.1),
                                                                        (8, nan)]:
        b = list(good)
        b[j] = v
        assert call(rows=(good, b)) == -1, (j, v)
    for j in range(3):
        b = list(good)
        b[3 + j] = b[j]
        assert call(rows=(b,)) == -1
    # edges that are valid: p_loss 0 and 1, zero excess and spread
    assert call(rows=([0, 0, 0, 10, 10, 3, 0.0, 0.0, 0.0], [0, 0, 0, 10, 10, 3, 0.0, 0.0, 1.0])) == 0
    with pytest.raises(L.KfposError):
        synth.toa_montecarlo_chunk(16, 0, 2, anc, DEV, obstacles=[[1, 1, 0, 0, 2, 3, 0, 0, 0]])


def test_sync_rule():
    """Device outputs leave the call asynchronous; host outputs are staged and the stream is synchronised."""
    import torch
    from tests.test_gpu_staging import _busy_after
    N, M, T = 1 << 16, 8, 20
    s = torch.cuda.Stream()
    sp = C.c_void_p(s.cuda_stream)
    anc = np.ascontiguousarray(synth.anchors_for(M))
    t = np.arange(1, T + 1) * 0.1
    gen = L.KfposSynthToa(seed=9, tag_z=1.0, sigma_r=0.1)
    tbl = table(STUDY)
    d_r = torch.empty((T, M, N), dtype=torch.int32, device=DEV)
    d_m = torch.empty((T, N), dtype=torch.int32, device=DEV)
    h_r = np.zeros((T, M, N), dtype=np.int32)
    h_m = np.zeros((T, N), dtype=np.uint32)

    def run(r, m):
        return lambda: L.check(L.lib().kfpos_synth_toa_ranges_geo(0, N, M, C.c_void_p(anc.ctypes.data), T,
                                                                  C.c_void_p(t.ctypes.data), C.byref(gen), 3,
                                                                  C.cast(tbl, C.c_void_p), L.FMT_I32_MM, r, m, sp),
                               "geo")
    dp = lambda x: C.c_void_p(x.data_ptr())
    hp = lambda x: C.c_void_p(x.ctypes.data)
    assert _busy_after(run(dp(d_r), dp(d_m)), s)
    assert _busy_after(run(dp(d_r), None), s)
    assert not _busy_after(run(hp(h_r), hp(h_m)), s)
    assert not _busy_after(run(dp(d_r), hp(h_m)), s)
    assert np.array_equal(h_r, d_r.cpu().numpy())
    assert np.array_equal(h_m, d_m.cpu().numpy().view(np.uint32))
    torch.cuda.synchronize()
