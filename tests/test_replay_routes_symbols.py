"""The route table of tests/replay_routes.py against the replay kernels the built library defines: every
instantiation of t6_replay_kernel, k8_replay_kernel and t9_replay_kernel is one row's tuple with (ES, EH) one of
(off, off), (on, off), (on, on), and every such name exists.  A new launcher route without a row fails here, and
so does a row that names a kernel the library does not have.  No GPU needed."""
import os
import re
import shutil
import subprocess

import pytest

from roskfpos_b200.lib import SO_PATH as LIB
from tests.replay_routes import ROUTES, STATS, TEMPLATE_ARGS

SYM = re.compile(r"\b(?:kfpos::)?((?:t6|k8|t9)_replay_kernel<[^<>]*>)")


def library_instantiations():
    if not os.path.exists(LIB):
        pytest.fail(f"{LIB} is not built (make -C roskfpos_b200/csrc)")
    nm = shutil.which("nm")
    assert nm, "nm (binutils) is needed to read the library's symbols"
    out = subprocess.run([nm, "-C", "--defined-only", LIB], capture_output=True, text=True, check=True).stdout
    return {m.group(1) for line in out.splitlines() for m in [SYM.search(line)] if m}


def test_table_shape():
    """One row per route, 17 + 8 + 8, no two rows with one tuple, tuples as long as their template."""
    ids = [r.id for r in ROUTES]
    assert len(ids) == len(set(ids))
    counts = {mdl: sum(r.model == mdl for r in ROUTES) for mdl in ("T6", "K8", "T9")}
    assert counts == {"T6": 17, "K8": 8, "T9": 8}
    for r in ROUTES:
        assert len(r.tup) == len(TEMPLATE_ARGS[r.kernel]), r


def test_library_defines_exactly_the_table():
    got = library_instantiations()
    want = {r.symbol(es, eh) for r in ROUTES for es, eh in STATS}
    assert len(want) == 99
    assert not got - want, f"replay kernels without a route table row: {sorted(got - want)}"
    assert not want - got, f"route table rows the library does not define: {sorted(want - got)}"
    for k in TEMPLATE_ARGS:
        assert sum(s.startswith(k + "<") for s in got) == 3 * sum(r.kernel == k for r in ROUTES)
