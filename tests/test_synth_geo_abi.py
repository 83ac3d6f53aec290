"""The obstacle generator's ABI without a GPU: the ctypes mirror of kfpos_obstacle matches the C struct,
malformed boxes are refused before any device work, and kfpos_synth_toa_ranges_geo fails loudly instead of
computing on the CPU."""
import ctypes as C
import os
import subprocess

import numpy as np

from roskfpos_b200 import lib as L


def test_obstacle_struct_layout(tmp_path):
    """sizeof and every offsetof of the C struct, printed by a C program, equal the ctypes mirror's."""
    fields = [name for name, _ in L.KfposObstacle._fields_]
    src = tmp_path / "layout.c"
    src.write_text('#include "kfpos_b200.h"\n#include <stddef.h>\n#include <stdio.h>\n'
                   "int main(void) {\n"
                   '  printf("%zu %d\\n", sizeof(kfpos_obstacle), KFPOS_MAX_OBSTACLES);\n' +
                   "".join(f'  printf("%zu\\n", offsetof(kfpos_obstacle, {f}));\n' for f in fields) +
                   "  return 0;\n}\n")
    exe = tmp_path / "layout"
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Wextra", "-pedantic", "-Werror",
                           f"-I{os.path.dirname(L.HEADER_PATH)}", str(src), "-o", str(exe)])
    got = [int(v) for v in subprocess.check_output([str(exe)]).split()]
    assert got[:2] == [C.sizeof(L.KfposObstacle), L.MAX_OBSTACLES]
    assert got[2:] == [getattr(L.KfposObstacle, f).offset for f in fields]


def boxes(rows):
    tbl = (L.KfposObstacle * max(len(rows), 1))()
    for o, b in zip(tbl, rows):
        o.lo[:], o.hi[:] = b[0:3], b[3:6]
        o.excess_per_m, o.spread, o.p_loss = b[6], b[7], b[8]
    return tbl


def call(lib, tbl, n, out):
    anc = np.ascontiguousarray(np.zeros((4, 3)))
    t = np.array([0.1, 0.2])
    gen = L.KfposSynthToa(seed=1, tag_z=1.0, sigma_r=0.1, nlos_mean=0.8)
    return lib.kfpos_synth_toa_ranges_geo(0, 8, 4, C.c_void_p(anc.ctypes.data), 2, C.c_void_p(t.ctypes.data),
                                          C.byref(gen), n, None if tbl is None else C.cast(tbl, C.c_void_p),
                                          L.FMT_I32_MM, C.c_void_p(out.ctypes.data), None, None)


def test_synth_geo_without_gpu(kflib):
    """Without a CUDA device kfpos_synth_toa_ranges_geo returns KFPOS_ERR_CUDA and writes nothing."""
    import torch
    if torch.cuda.is_available():
        return
    out = np.zeros((2, 4, 8), dtype=np.int32)
    assert call(kflib.lib(), boxes([[1, 1, 0, 2, 2, 3, 0.5, 0.1, 0.1]]), 1, out) == -2
    assert call(kflib.lib(), None, 0, out) == -2
    assert not out.any()


def test_malformed_boxes_refused(kflib):
    """Box checks come before the device check, so they hold with or without a GPU (KFPOS_ERR_INVALID)."""
    good = [1.0, 1.0, 0.0, 2.0, 2.0, 3.0, 0.5, 0.1, 0.1]
    nan, inf = float("nan"), float("inf")
    bad = []
    for j in range(6):
        for v in (nan, inf, -inf):
            b = list(good); b[j] = v; bad.append(b)
    for j in range(3):
        b = list(good); b[3 + j] = b[j]; bad.append(b)        # lo == hi
        b = list(good); b[3 + j] = b[j] - 1.0; bad.append(b)  # lo > hi
    for j in (6, 7):
        for v in (-1e-9, nan, inf):
            b = list(good); b[j] = v; bad.append(b)
    for v in (-0.1, 1.1, nan):
        b = list(good); b[8] = v; bad.append(b)
    out = np.zeros((2, 4, 8), dtype=np.int32)
    lib = kflib.lib()
    for b in bad:
        assert call(lib, boxes([good, b]), 2, out) == -1, b
    assert call(lib, boxes([good]), -1, out) == -1
    assert call(lib, boxes([good] * (L.MAX_OBSTACLES + 1)), L.MAX_OBSTACLES + 1, out) == -1
    assert call(lib, None, 1, out) == -1
    assert not out.any()
