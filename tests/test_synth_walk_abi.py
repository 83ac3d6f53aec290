"""The random walk's and the truth-driven generator's ABI without a GPU: the ctypes mirror of struct
kfpos_synth_walk matches the C struct, malformed arguments are refused before any device work, and both calls
fail loudly instead of computing on the CPU."""
import ctypes as C
import os
import subprocess

import numpy as np

from roskfpos_b200 import lib as L


def test_walk_struct_layout(tmp_path):
    """sizeof and every offsetof of the C struct, printed by a C program, equal the ctypes mirror's."""
    fields = [name for name, _ in L.KfposSynthWalk._fields_]
    src = tmp_path / "layout.c"
    src.write_text('#include "kfpos_b200.h"\n#include <stddef.h>\n#include <stdio.h>\n'
                   "int main(void) {\n"
                   '  printf("%zu\\n", sizeof(struct kfpos_synth_walk));\n' +
                   "".join(f'  printf("%zu\\n", offsetof(struct kfpos_synth_walk, {f}));\n' for f in fields) +
                   "  return 0;\n}\n")
    exe = tmp_path / "layout"
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Wextra", "-pedantic", "-Werror",
                           f"-I{os.path.dirname(L.HEADER_PATH)}", str(src), "-o", str(exe)])
    got = [int(v) for v in subprocess.check_output([str(exe)]).split()]
    assert got[0] == C.sizeof(L.KfposSynthWalk)
    assert got[1:] == [getattr(L.KfposSynthWalk, f).offset for f in fields]


GOOD = dict(seed=1, first_filter=0, first_epoch=0, period=0.1, accel_sd=(0.5, 0.5, 0.0), v_max=(1.5, 1.5, np.inf),
            lo=(0.5, 0.5, 0.0), hi=(9.5, 9.5, 2.0), init=1)


def walk_struct(**kw):
    a = dict(GOOD, **kw)
    w = L.KfposSynthWalk(seed=a["seed"], first_filter=a["first_filter"], first_epoch=a["first_epoch"],
                         period=a["period"], init=a["init"])
    w.accel_sd[:], w.v_max[:], w.lo[:], w.hi[:] = a["accel_sd"], a["v_max"], a["lo"], a["hi"]
    return w


def call_walk(lib, n=8, T=2, state=True, truth=True, walk=True, **kw):
    st = np.zeros((6, 8))
    tr = np.zeros((max(T, 1), 3, 8))
    rc = lib.kfpos_synth_walk(0, n, T, C.byref(walk_struct(**kw)) if walk else None,
                              C.c_void_p(st.ctypes.data) if state else None,
                              C.c_void_p(tr.ctypes.data) if truth else None, None)
    assert not st.any() and not tr.any()
    return rc


def call_truth(lib, n=8, M=4, T=2, truth=True, fmt=L.FMT_I32_MM, boxes=0, table=None, box=((1, 1, 0), (2, 2, 3)),
               **kw):
    """kfpos_synth_toa_ranges_truth with `boxes` boxes from a one-box table (table=False: a NULL table)."""
    anc = np.ascontiguousarray(np.zeros((4, 3)))
    tr = np.ones((max(T, 1), 3, 8))
    out = np.zeros((max(T, 1), 4, 8), dtype=np.int32)
    gen = L.KfposSynthToa(**dict(dict(seed=1, tag_z=1.0, sigma_r=0.1, nlos_mean=0.8), **kw))
    tbl = (L.KfposObstacle * 1)()
    tbl[0].lo[:], tbl[0].hi[:] = box
    rc = lib.kfpos_synth_toa_ranges_truth(0, n, M, C.c_void_p(anc.ctypes.data), T,
                                          C.c_void_p(tr.ctypes.data) if truth else None, C.byref(gen), boxes,
                                          C.cast(tbl, C.c_void_p) if (boxes > 0 if table is None else table) else None,
                                          fmt, C.c_void_p(out.ctypes.data), None, None)
    assert not out.any()
    return rc


def test_without_gpu(kflib):
    """Without a CUDA device both calls return KFPOS_ERR_CUDA and write nothing."""
    import torch
    if torch.cuda.is_available():
        return
    lib = kflib.lib()
    assert call_walk(lib) == -2
    assert call_walk(lib, T=0) == -2
    assert call_walk(lib, T=0, init=0) == -2
    assert call_truth(lib) == -2
    assert call_truth(lib, boxes=1) == -2
    assert call_truth(lib, T=0) == -2


def test_walk_refusals(kflib):
    """Argument checks come before the device check, so they hold with or without a GPU (KFPOS_ERR_INVALID)."""
    lib = kflib.lib()
    nan, inf = float("nan"), float("inf")
    bad = [dict(n=0), dict(n=-1), dict(T=-1), dict(walk=False), dict(state=False), dict(truth=False),
           dict(first_filter=-1), dict(first_epoch=-1), dict(first_epoch=0xFFFFFFFF - 1),
           dict(period=0.0), dict(period=-0.1), dict(period=nan), dict(period=inf), dict(init=2), dict(init=-1)]
    for j in range(3):
        for v in (-0.1, nan, inf):
            a = list(GOOD["accel_sd"]); a[j] = v; bad.append(dict(accel_sd=a))
        for v in (0.0, -1.0, nan, -inf):
            a = list(GOOD["v_max"]); a[j] = v; bad.append(dict(v_max=a))
        for key in ("lo", "hi"):
            for v in (nan, inf, -inf):
                a = list(GOOD[key]); a[j] = v; bad.append({key: a})
        a = list(GOOD["hi"]); a[j] = GOOD["lo"][j]; bad.append(dict(hi=a))        # lo == hi
        a = list(GOOD["hi"]); a[j] = GOOD["lo"][j] - 1.0; bad.append(dict(hi=a))  # lo > hi
    for kw in bad:
        assert call_walk(lib, **kw) == -1, kw


def test_truth_generator_refusals(kflib):
    """kfpos_synth_toa_ranges_truth refuses what kfpos_synth_toa_ranges_geo refuses, and a NULL truth."""
    lib = kflib.lib()
    for kw in (dict(truth=False), dict(n=0), dict(M=0), dict(M=33), dict(T=-1), dict(fmt=L.FMT_F64_M),
               dict(p_missing=1.5), dict(p_nlos=-0.1), dict(sigma_r=-0.1), dict(p_nlos=0.1, nlos_mean=0.0),
               dict(first_filter=-1), dict(first_epoch=0xFFFFFFFF), dict(boxes=-1), dict(boxes=L.MAX_OBSTACLES + 1),
               dict(boxes=1, table=False), dict(boxes=1, box=((1, 1, 0), (2, 1, 3))),
               dict(boxes=1, box=((1, 1, 0), (2, float("nan"), 3)))):
        assert call_truth(lib, **kw) == -1, kw
