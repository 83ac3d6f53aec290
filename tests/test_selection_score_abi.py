"""The selection scorer's ABI without a GPU: kfpos_synth_toa_ranges_nlos fails loudly instead of computing on the
CPU, and the numpy reference scorer the GPU tests compare with counts hand-made cases as documented."""
import ctypes as C

import numpy as np

from roskfpos_b200 import lib as L
from roskfpos_b200.batch import selection_summary
from tests.test_gpu_selection_score import reference_scores


def test_synth_toa_nlos_without_gpu(kflib):
    """Without a CUDA device kfpos_synth_toa_ranges_nlos returns KFPOS_ERR_CUDA: there is no CPU path."""
    import torch
    if torch.cuda.is_available():
        return
    anc = np.ascontiguousarray(np.zeros((4, 3)))
    t = np.array([0.1, 0.2])
    out = np.zeros((2, 4, 8), dtype=np.int32)
    mask = np.zeros((2, 8), dtype=np.uint32)
    gen = L.KfposSynthToa(seed=1, tag_z=1.0, sigma_r=0.1, p_nlos=0.5, nlos_mean=0.8)
    rc = kflib.lib().kfpos_synth_toa_ranges_nlos(0, 8, 4, C.c_void_p(anc.ctypes.data), 2, C.c_void_p(t.ctypes.data),
                                                 C.byref(gen), L.FMT_I32_MM, C.c_void_p(out.ctypes.data),
                                                 C.c_void_p(mask.ctypes.data), None)
    assert rc == -2
    assert not out.any() and not mask.any()


def test_reference_leave_one_out():
    # one row, 4 filters, 4 anchors; filter 0 drops slot 2 (NLOS), 1 drops nothing (-1), 2 drops slot 0 (LOS),
    # 3 drops slot 3, which is not present: nothing is dropped
    r = np.array([[[5, 5, 5, 5], [5, 5, 5, 5], [5, 5, 5, 5], [5, 5, 5, 0]]], dtype=np.int32)  # [1][M=4][N=4]
    sel = np.array([[2, -1, 0, 3]], dtype=np.int32)
    nlos = np.array([[0b0100, 0b0010, 0, 0b1000]], dtype=np.uint32)  # filter 3's bit is on an absent ranging
    c = reference_scores(r, sel, nlos, "loo")
    # present 4 + 4 + 4 + 3; dropped 1 + 0 + 1 + 0; NLOS present 1 + 1 + 0 + 0; NLOS dropped 1
    assert c.tolist() == [[15, 2, 2, 1, 2, 1, 2, 1]]
    s = selection_summary(c, 4)
    assert s["detection"][0] == 0.5 and s["false_drop"][0] == 1 / 13
    assert s["clean"][0] == 0.5 and s["false_alarm"][0] == 0.5


def test_reference_masks_with_32_anchors():
    """variant 1 / 2: sel is the used mask; with 32 anchors a full mask is -1 and bit 31 is the sign bit."""
    M, N = 32, 3
    r = np.ones((1, M, N), dtype=np.uint16)
    full = np.int32(-1)
    no31 = np.int32(0x7FFFFFFF)  # slot 31 dropped
    sel = np.array([[full, no31, no31]], dtype=np.int32)
    nlos = np.array([[0, 1 << 31, 1 << 5]], dtype=np.uint32)
    c = reference_scores(r, sel, nlos, "mask")
    # filter 1 dropped its NLOS slot 31; filter 2 dropped slot 31 (LOS) and kept NLOS slot 5
    assert c.tolist() == [[96, 2, 2, 1, 2, 1, 2, 0]]


def test_reference_null_mask_and_absent_rangings():
    """A NULL mask: no ranging is NLOS.  A used mask that names absent rangings drops nothing more, and slots that
    are absent are never counted as dropped."""
    r = np.array([[[1.0, 0.0], [np.nan, 2.0], [3.0, -1.0]]])  # f64 metres [1][M=3][N=2]: NaN and <= 0 are absent
    sel = np.array([[0b111, 0b001]], dtype=np.int32)
    c = reference_scores(r, sel, None, "mask")
    # filter 0: present {0, 2}, used covers them; filter 1: present {1}, used {0} -> slot 1 dropped
    assert c.tolist() == [[3, 1, 0, 0, 0, 0, 1, 1]]
    # plain T6 ignores sel; leave-one-out of an absent slot drops nothing
    assert reference_scores(r, None, None, "none").tolist() == [[3, 0, 0, 0, 0, 0, 0, 0]]
    assert reference_scores(r, np.array([[1, 0]], dtype=np.int32), None, "loo").tolist() == [[3, 0, 0, 0, 0, 0, 0, 0]]
    s = selection_summary(np.zeros((1, 8), dtype=np.uint64), 2)
    assert np.isnan(s["detection"][0]) and np.isnan(s["clean"][0]) and s["false_alarm"][0] == 0.0
