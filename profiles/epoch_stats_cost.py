"""Cost of the per-epoch statistics (kfpos_batch_set_truth_traj): the replay with and without them, alternated.

Two cases, timed with CUDA events around the replay launch only (set_state outside the window), five alternations
of off / on each:
  t6      the headline step: 1 Mi T6 filters x 1000 epochs x 8 anchors, int32 range log resident on the device
  config3 the BASELINE config-3 K8 shape: 1 Mi filters, UWB + IMU + compass macro-steps (synth.MACRO_IMU_MAG),
          inputs made on the device by kfpos_synth_k8, truth of every TOA event by kfpos_synth_k8_truth
Also times one kfpos_batch_epoch_stats fold of all rows (the end-of-run reduction).  Prints one JSON object with
ms per step, the on / off ratio, the GPU's name and its power limit.

    python profiles/epoch_stats_cost.py [--out FILE] [--k8-macro 20] [--reps 5]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, power, clk = [s.strip() for s in q.stdout.splitlines()[0].split(",")]
    return dict(gpu=name, power_limit=power, sm_clock_max=clk)


def alternate(run, set_on, reps, stream):
    """run() is one timed replay; set_on(flag) switches the statistics.  Returns per-mode lists of ms."""
    import torch
    res = {False: [], True: []}
    for flag in (False, True):  # warm-up of both instantiations
        set_on(flag)
        run()
    torch.cuda.synchronize()
    for _ in range(reps):
        for flag in (False, True):
            set_on(flag)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            run(a, b)
            b.synchronize()
            res[flag].append(a.elapsed_time(b))
    return res


def summary(res):
    off, on = float(np.median(res[False])), float(np.median(res[True]))
    return dict(ms_off=off, ms_on=on, ratio=on / off, ms_off_all=res[False], ms_on_all=res[True])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--filters", type=int, default=1 << 20)
    ap.add_argument("--tsteps", type=int, default=1000)
    ap.add_argument("--k8-macro", type=int, default=20)
    args = ap.parse_args()
    import torch
    from roskfpos_b200 import lib as L, synth
    from roskfpos_b200.batch import Batch, epoch_summary

    if not torch.cuda.is_available():
        raise SystemExit("epoch_stats_cost.py: no CUDA device")
    dev = torch.device("cuda", 0)
    stream = torch.cuda.current_stream()
    out = dict(gpu_info(), reps=args.reps)
    N, T = args.filters, args.tsteps
    anc = synth.anchors_for(8)

    # ---- T6 headline
    ranges, x0, _ = synth.device_ranges_mm(N, T, anc, 0.1, dev, seed=synth.SEED + 1000)
    truth = synth.device_truth_traj(N, T, 0.1, dev, seed=synth.SEED + 1000)
    x0f = torch.zeros((6, N), device=dev, dtype=torch.float64)
    x0f[:3] = x0
    with Batch(L.MODEL_T6, N, anchors=anc, accel_noise=0.5) as b:
        def set_on(flag):
            b.set_truth_traj(truth if flag else None, stream=stream)

        def run(e0=None, e1=None):
            b.set_state(x0f, None, stream=stream)
            if e0 is not None:
                e0.record(stream)
            b.replay_toa(0.1, ranges, err=0.01, stream=stream)
            if e1 is not None:
                e1.record(stream)
        out["t6"] = summary(alternate(run, set_on, args.reps, stream))
        out["t6"].update(filters=N, epochs=T, anchors=8, fmt="int32 mm, device resident",
                         kernel="t6_replay_kernel<false,false,8,false,1,ES>")
        set_on(True)
        run()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        st = b.epoch_stats(readback=False, stream=stream)
        e1.record(stream)
        e1.synchronize()
        out["t6"]["fold_ms"] = e0.elapsed_time(e1)
        s = epoch_summary(st.cpu().numpy())
        out["t6"].update(rmse_first=float(s["rmse"][0]), rmse_last=float(s["rmse"][-1]),
                         anees_last=float(s["anees"][-1]), n_last=float(s["n"][-1]))
    del ranges, truth

    # ---- config-3 K8
    w = synth.k8_montecarlo_chunk(N, 0, args.k8_macro, anc, dev, want_x0=True, want_truth_toa=True)
    with Batch(L.MODEL_K8, N, anchors=anc, xml=synth.K8_XML, accel_noise=0.5, jolt=0.5) as b:
        def set_on(flag):
            b.set_truth_traj(w["truth_toa"] if flag else None, stream=stream)

        def run(e0=None, e1=None):
            b.set_state(w["x0"], None, stream=stream)
            if e0 is not None:
                e0.record(stream)
            b.replay_events(w["events"], ranges=w["ranges"], sensors=w["sensors"], err=0.01, stream=stream)
            if e1 is not None:
                e1.record(stream)
        out["config3_k8"] = summary(alternate(run, set_on, args.reps, stream))
        out["config3_k8"].update(filters=N, macro_steps=args.k8_macro, events=w["n_events"], toa_rows=w["n_toa"],
                                 kernel="k8_replay_kernel<false,8,false,false,ES>")
        set_on(True)
        run()
        s = epoch_summary(b.epoch_stats())
        out["config3_k8"].update(rmse_last=float(s["rmse"][-1]), anees_last=float(s["anees"][-1]))
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
