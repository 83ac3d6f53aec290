"""Cost of the device-side ranging generator (kfpos_synth_toa_ranges) and what its inputs show.

Timed with CUDA events around the launches only, cases alternated within each repetition (median of --reps):
  generator  1 Mi filters x 1000 epochs x 8 anchors into a resident log: int32 and uint16 mm, plain and impaired
             (p_missing = p_nlos = 0.05); ms, G rangings/s, bytes written per second and their share of the
             7.7 TB/s HBM3e data-sheet bandwidth of one B200
  headline   the same generated int32 log replayed by T6 (the bench's T6 shape: 8 anchors, err 0.01,
             accel_noise 0.5), alternated with its generation: the generation share of generate + replay
  chunked    1 Mi filters x 10 000 epochs in chunks of 1000 (a resident int32 log would be 335 GB): generation
             and replay ms per chunk, the generation share
  accuracy   T6, 8 anchors, p_nlos 0.05, nlos_mean 0.8, 64 Ki filters x 1000 epochs through synth.toa_montecarlo:
             final RMSE and mean ANEES(t) for no selection, leave-one-out, variant 1 (n = 1), variant 2; the
             filters are told the true LOS noise (errorEstimation 0.10 m = sigma_r), so ANEES ~ 3 is consistent
Prints one JSON object with the GPU's name and power limit.

    python profiles/synth_toa_cost.py [--out FILE] [--reps 5]
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

HBM_BYTES_PER_S = 7.7e12  # NVIDIA HGX B200 data sheet, one GPU


def timed(fn, stream):
    import torch
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(stream)
    fn()
    b.record(stream)
    b.synchronize()
    return a.elapsed_time(b)


def alternate(cases, reps, stream):
    """cases: name -> fn.  One warm-up of each, then `reps` rounds over all cases.  Returns name -> [ms]."""
    import torch
    for fn in cases.values():
        fn()
    torch.cuda.synchronize()
    res = {k: [] for k in cases}
    for _ in range(reps):
        for k, fn in cases.items():
            res[k].append(timed(fn, stream))
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--filters", type=int, default=1 << 20)
    ap.add_argument("--epochs", type=int, default=1000)
    ap.add_argument("--long-epochs", type=int, default=10000)
    ap.add_argument("--acc-filters", type=int, default=1 << 16)
    ap.add_argument("--acc-err", type=float, default=0.10, help="errorEstimation of the accuracy runs, m")
    args = ap.parse_args()
    import torch
    from roskfpos_b200 import lib as L, synth
    from roskfpos_b200.batch import Batch, epoch_summary

    if not torch.cuda.is_available():
        raise SystemExit("synth_toa_cost.py: no CUDA device")
    dev = torch.device("cuda", 0)
    stream = torch.cuda.current_stream()
    out = dict(gpu_info(), reps=args.reps)
    N, T, M = args.filters, args.epochs, 8
    anc = synth.anchors_for(M)
    rangings = N * T * M
    imp = dict(p_missing=0.05, p_nlos=0.05)

    # ---- generator alone
    bufs = {L.FMT_I32_MM: {}, L.FMT_U16_MM: {}}

    def gen(fmt, **kw):
        return lambda: synth.toa_montecarlo_chunk(N, 0, T, anc, dev, fmt=fmt, out=bufs[fmt], stream=stream, **kw)
    cases = {"i32": gen(L.FMT_I32_MM), "i32_impaired": gen(L.FMT_I32_MM, **imp),
             "u16": gen(L.FMT_U16_MM), "u16_impaired": gen(L.FMT_U16_MM, **imp)}
    res = alternate(cases, args.reps, stream)
    g = {}
    for k, v in res.items():
        ms = float(np.median(v))
        nbytes = rangings * (2 if k.startswith("u16") else 4)
        g[k] = dict(ms=ms, ms_all=v, g_rangings_per_s=rangings / ms / 1e6, bytes_written=nbytes,
                    write_gb_per_s=nbytes / ms / 1e6, write_share_of_hbm=nbytes / (ms * 1e-3) / HBM_BYTES_PER_S)
    out["generator"] = dict(filters=N, epochs=T, anchors=M, impaired=imp, cases=g,
                            note="includes kfpos_synth_k8_truth of the final truth (one time, 24 MB)")
    del bufs[L.FMT_U16_MM]
    torch.cuda.empty_cache()

    # ---- the headline T6 shape on the generated log, alternated with its generation
    w = synth.toa_montecarlo_chunk(N, 0, T, anc, dev, want_x0=True, out=bufs[L.FMT_I32_MM], stream=stream)
    with Batch(L.MODEL_T6, N, anchors=anc, accel_noise=0.5) as b:
        def replay():
            b.replay_toa(w["dt"], w["ranges"], err=0.01, stream=stream)

        def reset():  # outside the timed windows
            b.set_state(w["x0"], None, stream=stream)
        gen_i32 = gen(L.FMT_I32_MM)
        for f in (reset, replay):
            f()
        torch.cuda.synchronize()
        gms, rms = [], []
        for _ in range(args.reps):
            gms.append(timed(gen_i32, stream))
            reset()
            rms.append(timed(replay, stream))
        x, _, st = b.get_state(want_P=False)
        tr = w["truth_end"].cpu().numpy()
        e = np.sqrt(((x[:3] - tr) ** 2).sum(axis=0))
        gm, rm = float(np.median(gms)), float(np.median(rms))
        out["headline"] = dict(filters=N, epochs=T, anchors=M, gen_ms=gm, replay_ms=rm, gen_share=gm / (gm + rm),
                               gen_ms_all=gms, replay_ms_all=rms, kernel="t6_replay_kernel, int32 log resident",
                               final_rmse=float(np.sqrt((e ** 2).mean())), n_status_bad=int((st != 0).sum()))

        # ---- chunked long run: generate chunk c, replay it, continue
        TL = args.long_epochs
        b.set_state(w["x0"], None, stream=stream)
        cg, cr = [], []
        for k0 in range(0, TL, T):
            n = min(T, TL - k0)
            wc = {}
            cg.append(timed(lambda: wc.update(synth.toa_montecarlo_chunk(N, k0, n, anc, dev, out=bufs[L.FMT_I32_MM],
                                                                         stream=stream)), stream))
            cr.append(timed(lambda: b.replay_toa(wc["dt"], wc["ranges"], err=0.01, stream=stream), stream))
        x, _, st = b.get_state(want_P=False)
        tr = wc["truth_end"].cpu().numpy()
        e = np.sqrt(((x[:3] - tr) ** 2).sum(axis=0))
        gm, rm = float(np.median(cg)), float(np.median(cr))
        out["chunked"] = dict(filters=N, epochs=TL, chunk=T, resident_log_gb=N * TL * M * 4 / 1e9,
                              gen_ms_per_chunk=gm, replay_ms_per_chunk=rm, gen_share=sum(cg) / (sum(cg) + sum(cr)),
                              total_ms=sum(cg) + sum(cr), gen_ms_all=cg, replay_ms_all=cr,
                              final_rmse=float(np.sqrt((e ** 2).mean())), n_status_bad=int((st != 0).sum()))
    del w, wc, bufs
    torch.cuda.empty_cache()

    # ---- accuracy of the NLOS modes on one generated workload
    NA = args.acc_filters
    modes = {"none": {}, "leave_one_out": dict(ignore_worst_anchor=1),
             "variant1_n1": dict(variant=1, num_ignored_rangings=1), "variant2": dict(variant=2)}
    acc = {}
    for name, cfg in modes.items():
        with Batch(L.MODEL_T6, NA, anchors=anc, accel_noise=0.5, **cfg) as b:
            rows = {}
            ms = timed(lambda: rows.update(r=synth.toa_montecarlo(b, T, T, anc, p_nlos=0.05, nlos_mean=0.8,
                                                                  err=args.acc_err, stream=stream)), stream)
            s = epoch_summary(rows["r"])
            acc[name] = dict(final_rmse=float(s["rmse"][-1]), final_rmse_xy=float(s["rmse_xy"][-1]),
                             mean_anees=float(np.nanmean(s["anees"])), final_anees=float(s["anees"][-1]),
                             n_bad_last=float(s["n_bad"][-1]), run_ms=ms)
    out["accuracy"] = dict(filters=NA, epochs=T, anchors=M, p_nlos=0.05, nlos_mean=0.8, sigma_r=0.10, err=args.acc_err,
                           modes=acc)
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
