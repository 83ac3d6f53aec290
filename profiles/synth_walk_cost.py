"""Cost of the random walk (kfpos_synth_walk) and of the truth-driven ranging generator (kfpos_synth_toa_ranges_truth).

Timed with CUDA events around the calls only, cases alternated within each repetition (median of --reps), at
1 Mi filters x 1000 epochs x 8 int32 anchors, sigma_r 0.10 m:
  walk       the room walk of DESIGN §4.5g, one Box-Muller pair per filter and epoch (accel_sd_z = 0), and the same
             walk with accel_sd_z > 0 (two pairs): the same bytes, twice the normals
  truth      the truth-driven generator from that walk: plain, impaired (5 % missing, 5 % NLOS), 3 study boxes
  lissajous  the Lissajous generator (kfpos_synth_toa_ranges / _geo) on the same shapes
  copy       a device-to-device cudaMemcpyAsync and a cudaMemsetAsync of the bytes the kernels move, the HBM yardsticks
Also the ptxas registers and spills of synth_walk_kernel and of the TRUTH instantiations.  Prints one JSON object
with the GPU's name, power limit and max SM clock.

    python profiles/synth_walk_cost.py [--out FILE] [--reps 5]
"""
from __future__ import annotations

import argparse
import json
import os
import re
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from epoch_stats_cost import gpu_info  # noqa: E402
from synth_geo_cost import STUDY  # noqa: E402
from synth_toa_cost import alternate  # noqa: E402

INF = float("inf")
ROOM_WALK = dict(accel_sd=(0.5, 0.5, 0.0), v_max=(1.5, 1.5, INF), lo=(0.5, 0.5, 0.5), hi=(9.5, 9.5, 1.5))


def ptxas_counts():
    """Registers and spill bytes of synth_walk_kernel and the TRUTH synth_toa_kernel instantiations."""
    path = os.path.join(ROOT, "roskfpos_b200", "csrc", "kfpos_synth.ptxas.log")
    if not os.path.exists(path):
        return None
    out, name = {}, None
    for line in open(path):
        m = re.search(r"Function properties for \S*synth_toa_kernelI([it])Lb(\d)ELb(\d)ELb(\d)ELb1E", line)
        if m:
            name = "synth_toa_kernel<%s, IMPAIR %s, MASK %s, GEO %s, TRUTH 1>" % (
                ("int32", "uint16")[m.group(1) == "t"], m.group(2), m.group(3), m.group(4))
            continue
        if re.search(r"Function properties for \S*synth_walk_kernel", line):
            name = "synth_walk_kernel"
            continue
        if re.search(r"Function properties for", line):
            name = None
            continue
        m = re.search(r"(\d+) bytes spill stores, (\d+) bytes spill loads", line)
        if m and name:
            out.setdefault(name, {})["spill_bytes"] = int(m.group(1)) + int(m.group(2))
        m = re.search(r"Used (\d+) registers", line)
        if m and name:
            out.setdefault(name, {})["registers"] = int(m.group(1))
            name = None
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--filters", type=int, default=1 << 20)
    ap.add_argument("--epochs", type=int, default=1000)
    args = ap.parse_args()
    import torch
    from roskfpos_b200 import synth

    if not torch.cuda.is_available():
        raise SystemExit("synth_walk_cost.py: no CUDA device")
    dev = torch.device("cuda", 0)
    stream = torch.cuda.current_stream()
    out = dict(gpu_info(), reps=args.reps, ptxas=ptxas_counts())
    N, T, M = args.filters, args.epochs, 8
    anc = synth.anchors_for(M)
    wb, gb = {}, {}
    wk = dict(seed=synth.SEED, period=0.1)
    # the truth every generator case reads: the room walk, made once outside the timed windows
    truth = synth.walk_truth_chunk(N, 0, T, dev, out=wb, stream=stream, **wk, **ROOM_WALK)["truth"]
    walk_out = {}  # both walk cases write the same buffers
    imp = dict(p_missing=0.05, p_nlos=0.05, nlos_mean=0.8)

    def walk(z):
        w = dict(ROOM_WALK, accel_sd=(0.5, 0.5, 0.3 if z else 0.0))
        return lambda: synth.walk_truth_chunk(N, 0, T, dev, out=walk_out, stream=stream, **wk, **w)

    def gen(use_truth, **kw):
        return lambda: synth.toa_montecarlo_chunk(N, 0, T, anc, dev, out=gb, stream=stream,
                                                  truth=truth if use_truth else None, **kw)
    # HBM yardsticks: the walk writes 24 B per filter and epoch; the generator reads those 24 B and writes 32 B.
    # The memset writes the walk's bytes into the walk's own buffer; the copy reads half of them from the generator's
    # truth and writes them into the other half (the same traffic), so that no buffer is added
    walk_bytes = 24 * N * T
    walk(False)()
    dst = walk_out["truth"].view(-1)
    half = dst.numel() // 2
    cases = {"walk_1_pair": walk(False), "walk_2_pairs": walk(True),
             "truth_plain": gen(True), "truth_impaired": gen(True, **imp), "truth_3_boxes": gen(True, obstacles=STUDY),
             "lissajous_plain": gen(False), "lissajous_impaired": gen(False, **imp),
             "lissajous_3_boxes": gen(False, obstacles=STUDY),
             "memset_walk_bytes": lambda: dst.zero_(),
             "copy_walk_bytes": lambda: dst[:half].copy_(truth.view(-1)[half:2 * half])}
    res = alternate(cases, args.reps, stream)
    ms = {k: float(np.median(v)) for k, v in res.items()}
    out["cases"] = {k: dict(ms=ms[k], ms_all=v) for k, v in res.items()}
    gen_bytes = (24 + 4 * M) * N * T
    tbs = lambda b, k: b / (ms[k] * 1e-3) / 1e12
    out["shape"] = dict(filters=N, epochs=T, anchors=M, fmt="int32", sigma_r=0.10, walk=ROOM_WALK,
                        walk_bytes=walk_bytes, truth_generator_bytes=gen_bytes)
    out["rates_tb_s"] = dict(walk_1_pair=tbs(walk_bytes, "walk_1_pair"), walk_2_pairs=tbs(walk_bytes, "walk_2_pairs"),
                             memset=tbs(walk_bytes, "memset_walk_bytes"),
                             copy_read_plus_write=tbs(16 * half, "copy_walk_bytes"),
                             truth_plain=tbs(gen_bytes, "truth_plain"))
    out["ratios"] = dict(walk_2_over_1_pair=ms["walk_2_pairs"] / ms["walk_1_pair"],
                         walk_over_memset=ms["walk_1_pair"] / ms["memset_walk_bytes"],
                         truth_over_lissajous_plain=ms["truth_plain"] / ms["lissajous_plain"],
                         truth_over_lissajous_impaired=ms["truth_impaired"] / ms["lissajous_impaired"],
                         truth_over_lissajous_3_boxes=ms["truth_3_boxes"] / ms["lissajous_3_boxes"])
    out["note"] = ("each toa_montecarlo_chunk call also writes its truth_end: a [3][N] row slice with a truth array, "
                   "one kfpos_synth_k8_truth time for the Lissajous; the walk's bytes are its truth stores (its "
                   "[6][N] state is 0.1 % of them)")
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
