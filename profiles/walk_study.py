"""The NLOS selection study of DESIGN §4.5d / §4.5e rerun on random walks that cover the whole site (DESIGN §4.5g).

Settings of §4.5d: 64 Ki filters x 1000 epochs, 8 int32 anchors, sigma_r 0.10 m with errorEstimation 0.10 m, 5 %
i.i.d. NLOS of mean 0.8 m, no missing rangings, no boxes.  Trajectories:
  lissajous  the fixed path of §4.5c-e (tag_z 1.0), rerun here so that every row comes from one build and one card
  room       the 8-anchor 10 x 10 m room, a walk over [0.5, 9.5]^2 x {1.0}, accel_sd (0.5, 0.5, 0) m/s^2,
             v_max (1.5, 1.5, inf) m/s
  corridor   40 m x 3 m with 8 wall anchors (INTEGRATION.md), the same walk over [0.5, 39.5] x [0.5, 2.5] x {1.0}
Modes: T6 plain, T6 leave-one-out, T6 variant 1 (one ranging ignored) and ML variant 1: the final RMSE, the mean
ANEES (T6), the detection and false-drop rates, and the PRESENT / LOS / USED floors (mean over the epochs and at
the final epoch); the wall time of each run (generation, replay, statistics, scores and floors).  Also how much of
the site each trajectory covers.  Prints one JSON object with the GPU's name, power limit and max SM clock.

    python profiles/walk_study.py [--out FILE] [--filters 65536] [--epochs 1000]
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from epoch_stats_cost import gpu_info  # noqa: E402
from selection_score_cost import rates  # noqa: E402

INF = float("inf")
SETS = ("present", "los", "used")
ROOM_WALK = dict(accel_sd=(0.5, 0.5, 0.0), v_max=(1.5, 1.5, INF), lo=(0.5, 0.5, 0.5), hi=(9.5, 9.5, 1.5))
# the corridor of INTEGRATION.md: anchors on both long walls, heights alternating so that the 3-D solve is posed
CORRIDOR_ANCHORS = np.array([[x, y, z] for y, zs in ((0.0, (2.5, 0.5)), (3.0, (0.5, 2.5)))
                             for x, z in zip((0.0, 40.0 / 3, 80.0 / 3, 40.0), zs * 2)])
CORRIDOR_WALK = dict(accel_sd=(0.5, 0.5, 0.0), v_max=(1.5, 1.5, INF), lo=(0.5, 0.5, 0.5), hi=(39.5, 2.5, 1.5))
T6_MODES = {"t6_none": {}, "t6_leave_one_out": dict(ignore_worst_anchor=1),
            "t6_variant1_n1": dict(variant=1, num_ignored_rangings=1)}


def floors(cr):
    from roskfpos_b200.batch import crlb_summary
    f = {}
    for s in SETS:
        c = crlb_summary(cr[s])
        f["mean_floor_" + s] = float(np.nanmean(c["rmse_bound"]))
        f["final_floor_" + s] = float(c["rmse_bound"][-1])
    return f


def coverage(truth, lo, hi, cell=0.5):
    """Share of the 0.5 m x-y cells of [lo, hi] the tags visit, and the share of positions within 0.5 m of a wall."""
    x, y = truth[:, 0].ravel(), truth[:, 1].ravel()
    nx, ny = int(np.ceil((hi[0] - lo[0]) / cell)), int(np.ceil((hi[1] - lo[1]) / cell))
    h, _, _ = np.histogram2d(x, y, bins=(nx, ny), range=((lo[0], hi[0]), (lo[1], hi[1])))
    near = (x < lo[0] + 0.5) | (x > hi[0] - 0.5) | (y < lo[1] + 0.5) | (y > hi[1] - 0.5)
    return dict(cells_visited=float((h > 0).mean()), min_cell_share=float(h.min() / h.sum()),
                max_cell_share=float(h.max() / h.sum()), near_wall=float(near.mean()))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--filters", type=int, default=1 << 16)
    ap.add_argument("--epochs", type=int, default=1000)
    args = ap.parse_args()
    import torch
    from roskfpos_b200 import lib as L, synth
    from roskfpos_b200.batch import Batch, epoch_summary

    if not torch.cuda.is_available():
        raise SystemExit("walk_study.py: no CUDA device")
    dev = torch.device("cuda", 0)
    stream = torch.cuda.current_stream()
    N, T = args.filters, args.epochs
    kw = dict(sigma_r=0.10, p_nlos=0.05, nlos_mean=0.8, tag_z=1.0)
    var = 0.10 ** 2 + 1e-6 / 12
    scenes = {"lissajous": (synth.anchors_for(8), None, (1.0, 1.0, 4.0)),
              "room": (synth.anchors_for(8), ROOM_WALK, (1.0, 1.0, 4.0)),
              "corridor": (CORRIDOR_ANCHORS, CORRIDOR_WALK, (20.0, 1.5, 1.5))}
    out = dict(gpu_info(), filters=N, epochs=T, anchors=8, err=0.10, var=var, **kw, scenes={})
    for scene, (anc, walk, start) in scenes.items():
        res = dict(anchors=anc.tolist(), walk=walk, ml_start=start, modes={})
        # the truth of the scene, for its coverage and for the ML runs
        if walk is None:
            wc = synth.toa_montecarlo_chunk(N, 0, T, anc, dev, want_truth=True, want_nlos=True, stream=stream, **kw)
            lo, hi = (0.5, 0.5), (9.5, 9.5)
        else:
            wt = synth.walk_truth_chunk(N, 0, T, dev, seed=synth.SEED, period=0.1, stream=stream, **walk)
            wc = synth.toa_montecarlo_chunk(N, 0, T, anc, dev, want_truth=True, want_nlos=True, stream=stream,
                                            truth=wt["truth"], **kw)
            lo, hi = walk["lo"], walk["hi"]
        res["coverage"] = coverage(wc["truth"].cpu().numpy(), lo, hi)
        for name, cfg in T6_MODES.items():
            with Batch(L.MODEL_T6, N, anchors=anc, accel_noise=0.5, **cfg) as b:
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                rows, sc, cr = synth.toa_montecarlo(b, T, T, anc, err=0.10, stream=stream, score=True, crlb=SETS,
                                                    walk=walk, **kw)
                torch.cuda.synchronize()
                wall = time.perf_counter() - t0
            s = epoch_summary(rows)
            res["modes"][name] = dict(final_rmse=float(s["rmse"][-1]), final_rmse_xy=float(s["rmse_xy"][-1]),
                                      mean_anees=float(np.nanmean(s["anees"])), run_s=wall, **rates(sc, N),
                                      **floors(cr))
        with Batch(L.MODEL_ML, N, anchors=anc, variant=1, num_ignored_rangings=1, ml_start=start) as b:
            o = dict(pos=torch.empty((3, N), dtype=torch.float64, device=dev),
                     sel=torch.empty((2, N), dtype=torch.int32, device=dev),
                     status=torch.empty(N, dtype=torch.int32, device=dev))
            c = torch.empty((T, L.SCORE_COLS), dtype=torch.int64, device=dev)
            cr = {s: torch.empty((T, L.CRLB_COLS), dtype=torch.float64, device=dev) for s in SETS}
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for k in range(T):
                b.ml_solve(wc["ranges"][k], err=0.10, out=o, stream=stream)
                b.score_selection(wc["ranges"][k], o["sel"], wc["nlos"][k], out=c[k:k + 1], stream=stream)
                for s in SETS:
                    b.crlb(wc["truth"][k], wc["ranges"][k], var, o["sel"], wc["nlos"][k], set=s,
                           out=cr[s][k:k + 1], stream=stream)
            torch.cuda.synchronize()
            wall = time.perf_counter() - t0
            e2 = ((o["pos"] - wc["truth"][-1]) ** 2).sum(dim=0)
            e2 = e2[torch.isfinite(e2)]
            res["modes"]["ml_variant1_n1"] = dict(final_rmse=float(torch.sqrt(e2.mean())), mean_anees=None,
                                                  run_s=wall, **rates(c.cpu().numpy().astype(np.uint64), N),
                                                  **floors({s: cr[s].cpu().numpy() for s in SETS}))
        out["scenes"][scene] = res
        del wc
        torch.cuda.empty_cache()
        print(scene, json.dumps(res["modes"]), flush=True)
    out["ml_note"] = ("ML batches solve each epoch alone from ml_start; final RMSE = the last epoch's estimates "
                      "against its truth; no covariance, so no ANEES; its run_s excludes generation")
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
