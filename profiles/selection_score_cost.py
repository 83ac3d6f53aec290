"""Cost of the NLOS detection scores (kfpos_synth_toa_ranges_nlos, kfpos_batch_score_selection) and what they show.

Timed with CUDA events around the calls only, variants alternated within each repetition (median of --reps):
  generator  1 Mi filters x 1000 epochs x 8 anchors, int32, p_missing = p_nlos = 0.05: the log alone and the log
             with its NLOS mask
  scorer     that log scored against the variant-1 selection of a T6 replay of it and the mask: ms, bytes read per
             second (n_rows N (M 4 + 4 + 4)), next to a device-to-device cudaMemcpyAsync of the same byte count
             (each byte read once and written once) timed in the same run
  replay     T6 leave-one-out and variant 1 (n = 1), 1 Mi filters x 100 epochs of the same log, with and without
             the `sel` output
  accuracy   8 anchors, 64 Ki filters x 1000 epochs, sigma_r 0.10 m with errorEstimation 0.10 m, 5 % NLOS of mean
             0.8 m (DESIGN §4.5c): final RMSE and the mean over the epochs of the detection, false-drop,
             clean-filter and false-alarm rates (batch.selection_summary) for T6 none / leave-one-out / variant 1 /
             variant 2 (synth.toa_montecarlo(score=True)) and ML variant 1 (n = 1) / variant 2, epoch by epoch
Prints one JSON object with the GPU's name, power limit and max SM clock.

    python profiles/selection_score_cost.py [--out FILE] [--reps 5]
"""
from __future__ import annotations

import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from epoch_stats_cost import gpu_info  # noqa: E402
from synth_toa_cost import alternate, timed  # noqa: E402

HBM_BYTES_PER_S = 7.7e12  # NVIDIA HGX B200 data sheet, one GPU


def rates(counts, n):
    from roskfpos_b200.batch import selection_summary
    s = selection_summary(counts, n)
    return {k: float(np.nanmean(v)) if np.isfinite(v).any() else float("nan") for k, v in s.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--filters", type=int, default=1 << 20)
    ap.add_argument("--epochs", type=int, default=1000)
    ap.add_argument("--replay-epochs", type=int, default=100)
    ap.add_argument("--acc-filters", type=int, default=1 << 16)
    args = ap.parse_args()
    import torch
    from roskfpos_b200 import lib as L, synth
    from roskfpos_b200.batch import Batch, epoch_summary

    if not torch.cuda.is_available():
        raise SystemExit("selection_score_cost.py: no CUDA device")
    dev = torch.device("cuda", 0)
    stream = torch.cuda.current_stream()
    out = dict(gpu_info(), reps=args.reps)
    N, T, M = args.filters, args.epochs, 8
    anc = synth.anchors_for(M)
    imp = dict(p_missing=0.05, p_nlos=0.05, nlos_mean=0.8)

    # ---- (a) generator with and without the mask
    bufs = {}
    gen = lambda nl: lambda: synth.toa_montecarlo_chunk(N, 0, T, anc, dev, out=bufs, stream=stream, want_nlos=nl,
                                                         **imp)
    res = alternate({"log": gen(False), "log_and_mask": gen(True)}, args.reps, stream)
    out["generator"] = dict(filters=N, epochs=T, anchors=M, impaired=imp, fmt="int32",
                            cases={k: dict(ms=float(np.median(v)), ms_all=v) for k, v in res.items()})
    out["generator"]["mask_cost"] = out["generator"]["cases"]["log_and_mask"]["ms"] / out["generator"]["cases"]["log"]["ms"]

    # ---- (b) the scorer on that log, next to a copy of the same byte count
    w = synth.toa_montecarlo_chunk(N, 0, T, anc, dev, out=bufs, stream=stream, want_nlos=True, want_x0=True, **imp)
    sel = torch.empty((T, N), dtype=torch.int32, device=dev)
    counts = torch.empty((T, L.SCORE_COLS), dtype=torch.int64, device=dev)
    with Batch(L.MODEL_T6, N, anchors=anc, accel_noise=0.5, variant=1, num_ignored_rangings=1) as b:
        b.set_state(w["x0"], None, stream=stream)
        b.replay_toa(w["dt"], w["ranges"], err=0.10, sel=sel, stream=stream)
        src = [w["ranges"], sel, w["nlos"]]
        dst = [torch.empty_like(x) for x in src]

        def copy():
            for d, s in zip(dst, src):
                d.copy_(s)
        score = lambda: b.score_selection(w["ranges"], sel, w["nlos"], out=counts, stream=stream)
        res = alternate({"score": score, "copy": copy}, args.reps, stream)
        nbytes = T * N * (M * 4 + 4 + 4)
        c = counts.cpu().numpy().astype(np.uint64)
    del dst
    sc, cp = float(np.median(res["score"])), float(np.median(res["copy"]))
    out["scorer"] = dict(filters=N, rows=T, anchors=M, fmt="int32", mode="T6 variant 1 (used mask)",
                         bytes_read=nbytes, ms=sc, ms_all=res["score"], read_gb_per_s=nbytes / sc / 1e6,
                         read_share_of_hbm_datasheet=nbytes / (sc * 1e-3) / HBM_BYTES_PER_S,
                         copy_ms=cp, copy_ms_all=res["copy"], copy_bytes=nbytes,
                         copy_gb_per_s=nbytes / cp / 1e6, score_over_copy=sc / cp,
                         datasheet_bound_ms=nbytes / HBM_BYTES_PER_S * 1e3, rates=rates(c, N),
                         note="copy_gb_per_s counts each copied byte once; the copy reads and writes it")

    # ---- (c) replays with and without the selection output
    TR = args.replay_epochs
    r100 = w["ranges"][:TR]
    rep = {}
    for name, cfg in (("leave_one_out", dict(ignore_worst_anchor=1)),
                      ("variant1_n1", dict(variant=1, num_ignored_rangings=1))):
        with Batch(L.MODEL_T6, N, anchors=anc, accel_noise=0.5, **cfg) as b:
            def run(with_sel):
                def f():
                    b.set_state(w["x0"], None, stream=stream)
                    b.replay_toa(w["dt"], r100, err=0.10, sel=sel[:TR] if with_sel else None, stream=stream)
                return f
            # set_state (a few MB of copies) sits inside both windows alike
            res = alternate({"without_sel": run(False), "with_sel": run(True)}, args.reps, stream)
        rep[name] = {k: dict(ms=float(np.median(v)), ms_all=v) for k, v in res.items()}
        rep[name]["ratio"] = rep[name]["with_sel"]["ms"] / rep[name]["without_sel"]["ms"]
    out["replay"] = dict(filters=N, epochs=TR, anchors=M, modes=rep)
    del w, bufs, sel, r100
    torch.cuda.empty_cache()

    # ---- (d) accuracy and detection, 64 Ki filters x 1000 epochs
    NA = args.acc_filters
    acc = {}
    t6_modes = {"t6_none": {}, "t6_leave_one_out": dict(ignore_worst_anchor=1),
                "t6_variant1_n1": dict(variant=1, num_ignored_rangings=1), "t6_variant2": dict(variant=2)}
    kw = dict(p_nlos=0.05, nlos_mean=0.8, sigma_r=0.10)
    for name, cfg in t6_modes.items():
        with Batch(L.MODEL_T6, NA, anchors=anc, accel_noise=0.5, **cfg) as b:
            rows, c = synth.toa_montecarlo(b, T, T, anc, err=0.10, score=True, stream=stream, **kw)
        s = epoch_summary(rows)
        acc[name] = dict(final_rmse=float(s["rmse"][-1]), **rates(c, NA))
    for name, cfg in (("ml_variant1_n1", dict(variant=1, num_ignored_rangings=1)), ("ml_variant2", dict(variant=2))):
        ch = {}
        with Batch(L.MODEL_ML, NA, anchors=anc, **cfg) as b:
            o = dict(pos=torch.empty((3, NA), dtype=torch.float64, device=dev),
                     sel=torch.empty((2, NA), dtype=torch.int32, device=dev),
                     status=torch.empty(NA, dtype=torch.int32, device=dev))
            c = torch.empty((T, L.SCORE_COLS), dtype=torch.int64, device=dev)
            wc = synth.toa_montecarlo_chunk(NA, 0, T, anc, dev, out=ch, want_truth=True, want_nlos=True,
                                            stream=stream, **kw)
            for k in range(T):
                b.ml_solve(wc["ranges"][k], err=0.10, out=o, stream=stream)
                b.score_selection(wc["ranges"][k], o["sel"], wc["nlos"][k], out=c[k:k + 1], stream=stream)
            e2 = ((o["pos"] - wc["truth"][-1]) ** 2).sum(dim=0)
            e2 = e2[torch.isfinite(e2)]
            acc[name] = dict(final_rmse=float(torch.sqrt(e2.mean())), **rates(c.cpu().numpy().astype(np.uint64), NA))
    out["accuracy"] = dict(filters=NA, epochs=T, anchors=M, err=0.10, modes=acc,
                           ml_note="ML batches solve each epoch alone from ml_start (1, 1, 4); final RMSE = the last "
                                   "epoch's estimates against its truth", **kw)
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
