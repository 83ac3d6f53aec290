"""The ranging generator's ABI without a GPU: the ctypes mirror of kfpos_synth_toa matches the C struct, and
kfpos_synth_toa_ranges fails loudly instead of computing on the CPU."""
import ctypes as C
import os
import subprocess

import numpy as np

from roskfpos_b200 import lib as L


def test_synth_toa_struct_layout(tmp_path):
    """sizeof and every offsetof of the C struct, printed by a C program, equal the ctypes mirror's."""
    fields = [name for name, _ in L.KfposSynthToa._fields_]
    src = tmp_path / "layout.c"
    src.write_text('#include "kfpos_b200.h"\n#include <stddef.h>\n#include <stdio.h>\n'
                   "int main(void) {\n"
                   '  printf("%zu\\n", sizeof(kfpos_synth_toa));\n' +
                   "".join(f'  printf("%zu\\n", offsetof(kfpos_synth_toa, {f}));\n' for f in fields) +
                   "  return 0;\n}\n")
    exe = tmp_path / "layout"
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Wextra", "-pedantic", "-Werror",
                           f"-I{os.path.dirname(L.HEADER_PATH)}", str(src), "-o", str(exe)])
    got = [int(v) for v in subprocess.check_output([str(exe)]).split()]
    assert got[0] == C.sizeof(L.KfposSynthToa)
    assert got[1:] == [getattr(L.KfposSynthToa, f).offset for f in fields]


def test_synth_toa_without_gpu(kflib):
    """Without a CUDA device kfpos_synth_toa_ranges returns KFPOS_ERR_CUDA: there is no CPU path."""
    import torch
    if torch.cuda.is_available():
        return
    anc = np.ascontiguousarray(np.zeros((4, 3)))
    t = np.array([0.1, 0.2])
    out = np.zeros((2, 4, 8), dtype=np.int32)
    gen = L.KfposSynthToa(seed=1, tag_z=1.0, sigma_r=0.1, nlos_mean=0.8)
    rc = kflib.lib().kfpos_synth_toa_ranges(0, 8, 4, C.c_void_p(anc.ctypes.data), 2, C.c_void_p(t.ctypes.data),
                                            C.byref(gen), L.FMT_I32_MM, C.c_void_p(out.ctypes.data), None)
    assert rc == -2
    assert not out.any()
