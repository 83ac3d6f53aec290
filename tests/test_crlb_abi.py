"""The Cramer-Rao bound's host side without a GPU: the numpy reference the GPU tests compare with, on hand-made
cases whose bound is known, the rank tree of sharded runs and the per-row summary."""
import numpy as np

from roskfpos_b200.batch import crlb_summary, rank_tree
from tests.test_gpu_crlb import reference_crlb, reference_terms

# tag at the origin, one anchor on each negative axis: g = e_x, e_y, e_z, so J = diag(1 / v)
AXES = np.array([(-1.0, 0, 0), (0, -2.0, 0), (0, 0, -3.0)])
ORIGIN = np.zeros((1, 3, 1))


def one(ranges_present, var=0.01, truth=ORIGIN, anc=AXES, dim=3, **kw):
    r = np.asarray(ranges_present, dtype=np.int32).reshape(1, -1, 1)
    return reference_crlb(truth, r, anc, var, dim, **kw)[0]


def test_axis_anchors_give_a_diagonal_information():
    v = np.array([0.01, 0.04, 0.09]).reshape(1, 3, 1)
    assert np.allclose(one([1, 1, 1], v), [0.14, 0.05, 1, 0], rtol=1e-15, atol=0)
    assert np.allclose(one([1, 1, 1], 0.01), [0.03, 0.02, 1, 0], rtol=1e-15, atol=0)
    # 2-D: the x-y part of the same unit vectors; the z anchor adds nothing to it
    assert np.allclose(one([1, 1, 1], v, dim=2), [0.05, 0.05, 1, 0], rtol=1e-15, atol=0)


def test_fewer_rangings_than_dimensions_have_no_bound():
    assert one([1, 1, 0]).tolist() == [0, 0, 0, 1]
    assert one([1, 0, 0], dim=2).tolist() == [0, 0, 0, 1]
    assert one([1, 1, 0], dim=2)[2] == 1
    # four anchors on one line through the tag: |S| >= D, J singular -> a zero pivot, no bound
    line = np.array([(-1.0, 0, 0), (-2.0, 0, 0), (1.0, 0, 0), (3.0, 0, 0)])
    assert one([1, 1, 1, 1], anc=line).tolist() == [0, 0, 0, 1]


def test_bad_variances_and_truths():
    for bad in (0.0, -0.01, np.nan, np.inf):
        v = np.array([0.01, bad, 0.01]).reshape(1, 3, 1)
        assert one([1, 1, 1], v).tolist() == [0, 0, 0, 1], bad
        # a bad variance of a ranging outside S is not read
        got = reference_crlb(ORIGIN, np.array([[[1], [1], [1]]], dtype=np.int32), AXES, v, 3, set="los",
                             nlos=np.array([[0b010]], dtype=np.uint32))
        assert got[0].tolist() == [0, 0, 0, 1]  # only 2 LOS rangings left
        four = np.vstack([AXES, [(1.0, 1.0, 1.0)]])
        v4 = np.array([0.01, bad, 0.01, 0.01]).reshape(1, 4, 1)
        got = reference_crlb(ORIGIN, np.ones((1, 4, 1), dtype=np.int32), four, v4, 3, set="los",
                             nlos=np.array([[0b0010]], dtype=np.uint32))
        assert got[0, 2] == 1, bad
    assert one([1, 1, 1], truth=np.array([[[np.nan], [0.0], [0.0]]])).tolist() == [0, 0, 0, 1]


def test_two_d_against_three_d():
    """Same anchors and tag: the 2-D information is the x-y block of the 3-D one, so its inverse is never larger
    than the x-y block of the 3-D inverse (a Schur complement)."""
    rng = np.random.default_rng(3)
    anc = np.column_stack([rng.uniform(0, 10, 6), rng.uniform(0, 10, 6), rng.uniform(0.3, 2.7, 6)])
    truth = np.stack([rng.uniform(2, 8, (5, 64)), rng.uniform(2, 8, (5, 64)), np.full((5, 64), 1.0)], axis=1)
    r = np.ones((5, 6, 64), dtype=np.int32)
    t3, _ = reference_terms(truth, r, anc, 0.01, 3)
    t2, _ = reference_terms(truth, r, anc, 0.01, 2)
    assert (t2[..., 0] == t2[..., 1]).all() and (t2[..., 2] == 1).all() and (t3[..., 2] == 1).all()
    assert (t2[..., 1] <= t3[..., 1] * (1 + 1e-12)).all() and (t3[..., 0] > t3[..., 1]).all()
    # anchors in the tag's horizontal plane: the 3-D J has no z information, the 2-D one is regular
    flat = np.array([(-1.0, 0, 0), (0, -1.0, 0), (1.0, 1.0, 0)])
    assert one([1, 1, 1], anc=flat).tolist() == [0, 0, 0, 1]
    assert one([1, 1, 1], anc=flat, dim=2)[2] == 1


def test_used_sets_and_32_anchor_masks():
    """sel read as the scorer reads it: leave-one-out slot, uint32 used mask (bit 31 = the sign bit)."""
    rng = np.random.default_rng(5)
    anc = np.column_stack([rng.uniform(0, 10, 32), rng.uniform(0, 10, 32), rng.uniform(0.3, 2.7, 32)])
    truth = np.array([[[5.0, 5.0, 5.0, 5.0], [5.0, 5.0, 5.0, 5.0], [1.0, 1.0, 1.0, 1.0]]])
    r = np.ones((1, 32, 4), dtype=np.uint16)
    sel = np.array([[-1, 0x7FFFFFFF, -1, 0x7FFFFFFF]], dtype=np.int32)
    t, _ = reference_terms(truth, r, anc, 0.01, 3, sel=sel, mode="mask", set="used")
    p, _ = reference_terms(truth, r, anc, 0.01, 3)
    assert (t[0, [0, 2], 0] == p[0, [0, 2], 0]).all() and (t[0, [1, 3], 0] > p[0, [1, 3], 0]).all()
    no31 = np.delete(np.arange(32), 31)
    q, _ = reference_terms(truth, r[:, no31], anc[no31], 0.01, 3)
    assert t[0, 1, 0] == q[0, 1, 0]
    loo = np.array([[31, -1, 40, 31]], dtype=np.int32)  # out-of-range slots drop nothing
    t, _ = reference_terms(truth, r, anc, 0.01, 3, sel=loo, mode="loo", set="used")
    assert t[0, 0, 0] == q[0, 0, 0] and t[0, 1, 0] == p[0, 1, 0] and t[0, 2, 0] == p[0, 2, 0]
    t, _ = reference_terms(truth, r, anc, 0.01, 3, sel=loo, mode="none", set="used")
    assert (t[..., 0] == p[..., 0]).all()


def test_rank_tree_is_the_pairwise_tree():
    a = np.array([[[0.1, 1.0]], [[0.2, 2.0]], [[0.3, 3.0]], [[1e16, 4.0]], [[-1e16, 5.0]]])  # [5 ranks][1 row][2]
    want = (((a[0] + a[1]) + (a[2] + a[3])) + a[4])[0]
    assert np.array_equal(rank_tree(a), want[None])
    assert np.array_equal(rank_tree(a[:3]), ((a[0] + a[1]) + a[2]))
    assert np.array_equal(rank_tree(a[:1]), a[0])
    assert np.array_equal(rank_tree(list(a[:2])), a[0] + a[1])
    b = np.array([1.0, 1e16, -1e16, 1.0]).reshape(4, 1, 1)  # the order is not the left-to-right sum's
    assert rank_tree(b)[0, 0] == 0.0 and ((b[0] + b[1]) + b[2]) + b[3] == 1.0
    try:
        rank_tree(np.zeros((0, 1, 4)))
    except ValueError:
        pass
    else:
        raise AssertionError("rank_tree accepted no ranks")


def test_summary_of_empty_rows():
    s = crlb_summary(np.array([[0.02, 0.01, 2.0, 1.0], [0.0, 0.0, 0.0, 3.0]]))
    assert np.allclose(s["rmse_bound"][:1], [0.1]) and np.allclose(s["rmse_xy_bound"][:1], [np.sqrt(0.005)])
    assert np.isnan(s["rmse_bound"][1]) and np.isnan(s["rmse_xy_bound"][1])
    assert s["n"].tolist() == [2.0, 0.0] and s["n_none"].tolist() == [1.0, 3.0]
