"""Per-epoch statistics without a GPU: the summary helper, and the handle-free entry point failing loudly."""
import ctypes as C

import numpy as np


def test_epoch_summary_rows():
    from roskfpos_b200.batch import epoch_summary
    s = np.array([[8.0, 2.0, 2.0, 1.0, 6.0, 2.0],
                  [0.0, 0.0, 0.0, 0.0, 0.0, 0.0]])
    out = epoch_summary(s)
    assert out["rmse"][0] == 2.0 and out["rmse_xy"][0] == 1.0 and out["anees"][0] == 3.0
    assert out["n"][0] == 2.0 and out["n_bad"][0] == 1.0
    assert np.isnan(out["rmse"][1]) and np.isnan(out["anees"][1]) and out["n"][1] == 0.0


def test_synth_truth_without_gpu(kflib):
    """kfpos_synth_k8_truth never computes on the CPU: without a CUDA device it returns KFPOS_ERR_CUDA."""
    import torch
    if torch.cuda.is_available():
        return
    t = np.array([0.1, 0.2])
    out = np.zeros((2, 3, 4))
    rc = kflib.lib().kfpos_synth_k8_truth(0, 4, 0, C.c_uint64(1), 2, C.c_void_p(t.ctypes.data), 1.0,
                                          C.c_void_p(out.ctypes.data), None)
    assert rc == -2
