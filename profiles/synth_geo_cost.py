"""Cost of obstacle-based NLOS in the ranging generator (kfpos_synth_toa_ranges_geo) and what it shows.

Timed with CUDA events around the calls only, cases alternated within each repetition (median of --reps):
  generator  1 Mi filters x 1000 epochs x 8 int32 anchors, sigma_r 0.10 m: the plain generator (with and without
             its i.i.d. mask) next to 3 (the study scenario), 8 and 32 boxes, with and without the mask; the ptxas
             registers and spills of the GEO instantiations
  headline   generation with the 3 study boxes + the T6 replay of the bench's shape (err 0.01, accel_noise 0.5)
  geometry   the study boxes at 4096 filters x 1000 epochs, sigma_r 0, p_loss 0 (the mask is then the blocked set):
             blocked fraction of the rangings, epochs with a blocked ranging, mean run length of a blocked
             (filter, anchor) pair in epochs, blocked fraction per anchor
  study      the six modes of DESIGN §4.5d / §4.5e on the study boxes: 8 anchors, 64 Ki filters x 1000 epochs,
             sigma_r 0.10 m with errorEstimation 0.10 m, tag_z 1.0, no i.i.d. NLOS: final RMSE, the detection,
             false-drop, clean-filter and false-alarm rates, the PRESENT / LOS / USED floors, mean ANEES (filters)
Prints one JSON object with the GPU's name, power limit and max SM clock.

    python profiles/synth_geo_cost.py [--out FILE] [--reps 5]
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
from selection_score_cost import rates  # noqa: E402
from synth_toa_cost import alternate, timed  # noqa: E402

SETS = ("present", "los", "used")
# DESIGN §4.5f: pillar, partition, metal cabinet (lo xyz, hi xyz, excess_per_m, spread, p_loss)
STUDY = np.array([[1.2, 7.6, 0.0, 1.8, 8.2, 3.0, 1.2, 0.2, 0.1],
                  [8.6, 2.0, 0.0, 8.75, 3.5, 2.2, 0.6, 0.1, 0.05],
                  [3.6, 8.4, 0.0, 4.6, 8.9, 1.2, 0.0, 1.0, 0.5]])


def boxes(n):
    """The study boxes, then seeded random boxes of 0.2-1.5 m on the floor of the 10 x 10 m room."""
    rng = np.random.default_rng(1234)
    extra = []
    for _ in range(max(n - len(STUDY), 0)):
        lo = np.array([rng.uniform(0, 9), rng.uniform(0, 9), 0.0])
        size = np.array([rng.uniform(0.2, 1.5), rng.uniform(0.2, 1.5), rng.uniform(0.8, 2.8)])
        extra.append(np.concatenate([lo, lo + size, [0.5, 0.2, 0.1]]))
    return np.vstack([STUDY] + extra)[:n] if extra else STUDY[:n]


def ptxas_counts():
    """Registers and spill bytes of the synth_toa_kernel instantiations, from the build's ptxas log."""
    path = os.path.join(ROOT, "roskfpos_b200", "csrc", "kfpos_synth.ptxas.log")
    if not os.path.exists(path):
        return None
    out, name = {}, None
    for line in open(path):
        m = re.search(r"Function properties for \S*synth_toa_kernelI([it])Lb(\d)ELb(\d)ELb(\d)E", line)
        if m:
            name = "synth_toa_kernel<%s, IMPAIR %s, MASK %s, GEO %s>" % (
                ("int32", "uint16")[m.group(1) == "t"], m.group(2), m.group(3), m.group(4))
            continue
        m = re.search(r"(\d+) bytes spill stores, (\d+) bytes spill loads", line)
        if m and name:
            out.setdefault(name, {})["spill_bytes"] = int(m.group(1)) + int(m.group(2))
        m = re.search(r"Used (\d+) registers", line)
        if m and name:
            out.setdefault(name, {})["registers"] = int(m.group(1))
            name = None
    return out


def run_lengths(blocked):
    """Mean length in epochs of the runs of consecutive blocked epochs, blocked [T][M][N]."""
    b = blocked.reshape(blocked.shape[0], -1).astype(np.int8)
    edges = np.diff(np.vstack([np.zeros((1, b.shape[1]), np.int8), b, np.zeros((1, b.shape[1]), np.int8)]), axis=0)
    n_runs = int((edges == 1).sum())
    return float(b.sum()) / n_runs if n_runs else float("nan")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--filters", type=int, default=1 << 20)
    ap.add_argument("--epochs", type=int, default=1000)
    ap.add_argument("--acc-filters", type=int, default=1 << 16)
    args = ap.parse_args()
    import torch
    from roskfpos_b200 import lib as L, synth
    from roskfpos_b200.batch import Batch, crlb_summary, epoch_summary

    if not torch.cuda.is_available():
        raise SystemExit("synth_geo_cost.py: no CUDA device")
    dev = torch.device("cuda", 0)
    stream = torch.cuda.current_stream()
    out = dict(gpu_info(), reps=args.reps, ptxas=ptxas_counts())
    N, T, M = args.filters, args.epochs, 8
    anc = synth.anchors_for(M)

    # ---- (a) the generator alone, 0 / 3 / 8 / 32 boxes, with and without the mask
    bufs = {}

    def gen(n_boxes, mask):
        return lambda: synth.toa_montecarlo_chunk(N, 0, T, anc, dev, out=bufs, stream=stream, want_nlos=mask,
                                                  obstacles=boxes(n_boxes) if n_boxes else None)
    cases = {f"{nb}_boxes{'_mask' if mask else ''}": gen(nb, mask) for nb in (0, 3, 8, 32) for mask in (False, True)}
    res = alternate(cases, args.reps, stream)
    g = {k: dict(ms=float(np.median(v)), ms_all=v) for k, v in res.items()}
    for k in g:
        base = g["0_boxes_mask" if k.endswith("_mask") else "0_boxes"]["ms"]
        g[k]["over_plain"] = g[k]["ms"] / base
    out["generator"] = dict(filters=N, epochs=T, anchors=M, fmt="int32", sigma_r=0.10, cases=g,
                            note="0 boxes is the plain generator (kfpos_synth_toa_ranges / _nlos); each call also "
                                 "computes the final truth (kfpos_synth_k8_truth, one time)")

    # ---- (b) generation with the study boxes + the headline T6 replay
    w = synth.toa_montecarlo_chunk(N, 0, T, anc, dev, want_x0=True, out=bufs, stream=stream, obstacles=STUDY)
    with Batch(L.MODEL_T6, N, anchors=anc, accel_noise=0.5) as b:
        def replay():
            b.replay_toa(w["dt"], w["ranges"], err=0.01, stream=stream)

        def reset():  # outside the timed windows
            b.set_state(w["x0"], None, stream=stream)
        gen3 = gen(3, False)
        for f in (gen3, reset, replay):
            f()
        torch.cuda.synchronize()
        gms, rms = [], []
        for _ in range(args.reps):
            gms.append(timed(gen3, stream))
            reset()
            rms.append(timed(replay, stream))
        gm, rm = float(np.median(gms)), float(np.median(rms))
        out["headline"] = dict(filters=N, epochs=T, anchors=M, boxes=3, gen_ms=gm, replay_ms=rm,
                               gen_share=gm / (gm + rm), gen_ms_all=gms, replay_ms_all=rms)
    del w, bufs
    torch.cuda.empty_cache()

    # ---- (c) the geometry of the study scenario
    NG = 4096
    geo0 = STUDY.copy()
    geo0[:, 8] = 0.0
    wg = synth.toa_montecarlo_chunk(NG, 0, T, anc, dev, sigma_r=0.0, want_nlos=True, obstacles=geo0, stream=stream)
    m = wg["nlos"].cpu().numpy().view(np.uint32)
    blocked = ((m[:, None, :] >> np.arange(M, dtype=np.uint32)[None, :, None]) & 1).astype(bool)  # [T][M][N]
    out["geometry"] = dict(filters=NG, epochs=T, period_s=0.1, blocked_fraction=float(blocked.mean()),
                           epochs_with_blocked=float(blocked.any(axis=1).mean()),
                           mean_run_epochs=run_lengths(blocked),
                           per_anchor=[float(v) for v in blocked.mean(axis=(0, 2))],
                           numpy_estimate=dict(blocked_fraction=0.116, epochs_with_blocked=0.79, mean_run_epochs=47,
                                               anchors_2_5_6=[0.21, 0.34, 0.32]))
    del wg, m, blocked

    # ---- (d) the six modes on the study boxes, 64 Ki filters x 1000 epochs
    NA = args.acc_filters
    kw = dict(sigma_r=0.10, p_nlos=0.0, tag_z=1.0)
    var = 0.10 ** 2 + 1e-6 / 12
    acc = {}

    def floors(cr):
        f = {}
        for s in SETS:
            c = crlb_summary(cr[s])
            f["mean_floor_" + s] = float(np.nanmean(c["rmse_bound"]))
            f["final_floor_" + s] = float(c["rmse_bound"][-1])
        return f
    t6_modes = {"t6_none": {}, "t6_leave_one_out": dict(ignore_worst_anchor=1),
                "t6_variant1_n1": dict(variant=1, num_ignored_rangings=1), "t6_variant2": dict(variant=2)}
    for name, cfg in t6_modes.items():
        with Batch(L.MODEL_T6, NA, anchors=anc, accel_noise=0.5, **cfg) as b:
            rows, sc, cr = synth.toa_montecarlo(b, T, T, anc, err=0.10, stream=stream, score=True, crlb=SETS,
                                                obstacles=STUDY, **kw)
        s = epoch_summary(rows)
        acc[name] = dict(final_rmse=float(s["rmse"][-1]), final_rmse_xy=float(s["rmse_xy"][-1]),
                         mean_anees=float(np.nanmean(s["anees"])), **rates(sc, NA), **floors(cr))
    for name, cfg in (("ml_variant1_n1", dict(variant=1, num_ignored_rangings=1)), ("ml_variant2", dict(variant=2))):
        ch = {}
        with Batch(L.MODEL_ML, NA, anchors=anc, **cfg) as b:
            o = dict(pos=torch.empty((3, NA), dtype=torch.float64, device=dev),
                     sel=torch.empty((2, NA), dtype=torch.int32, device=dev),
                     status=torch.empty(NA, dtype=torch.int32, device=dev))
            c = torch.empty((T, L.SCORE_COLS), dtype=torch.int64, device=dev)
            cr = {s: torch.empty((T, L.CRLB_COLS), dtype=torch.float64, device=dev) for s in SETS}
            wc = synth.toa_montecarlo_chunk(NA, 0, T, anc, dev, out=ch, want_truth=True, want_nlos=True,
                                            stream=stream, obstacles=STUDY, **kw)
            for k in range(T):
                b.ml_solve(wc["ranges"][k], err=0.10, out=o, stream=stream)
                b.score_selection(wc["ranges"][k], o["sel"], wc["nlos"][k], out=c[k:k + 1], stream=stream)
                for s in SETS:
                    b.crlb(wc["truth"][k], wc["ranges"][k], var, o["sel"], wc["nlos"][k], set=s,
                           out=cr[s][k:k + 1], stream=stream)
            e2 = ((o["pos"] - wc["truth"][-1]) ** 2).sum(dim=0)
            e2 = e2[torch.isfinite(e2)]
            acc[name] = dict(final_rmse=float(torch.sqrt(e2.mean())), mean_anees=None,
                             **rates(c.cpu().numpy().astype(np.uint64), NA),
                             **floors({s: cr[s].cpu().numpy() for s in SETS}))
    out["study"] = dict(filters=NA, epochs=T, anchors=M, err=0.10, var=var, boxes=STUDY.tolist(), modes=acc,
                        ml_note="ML batches solve each epoch alone from ml_start (1, 1, 4); final RMSE = the last "
                                "epoch's estimates against its truth; no covariance, so no ANEES", **kw)
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
