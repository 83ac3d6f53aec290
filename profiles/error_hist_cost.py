"""Cost of the per-epoch error histograms (kfpos_batch_set_error_hist): the replay with statistics off, with the
per-epoch statistics only (ES) and with statistics and histogram (ES + hist), alternated.

Two cases, timed with CUDA events around the replay launch only (set_state and the registrations outside the
window), --reps alternations of the three modes each:
  t6      the headline step: 1 Mi T6 filters x 1000 epochs x 8 anchors, int32 range log resident on the device,
          an ERR histogram of 200 edges (0.01 m steps)
  config3 the BASELINE config-3 K8 shape: 1 Mi filters, UWB + IMU + compass macro-steps (synth.MACRO_IMU_MAG),
          inputs made on the device by kfpos_synth_k8, truth of every TOA event by kfpos_synth_k8_truth, a NEES
          histogram
Also times one kfpos_batch_error_hist readback of all rows (into a device tensor and into host memory) and checks
that every row's total equals its epoch_stats count.  Prints one JSON object with ms per step, the ratios, the
GPU's name, its power limit and max SM clock.

    python profiles/error_hist_cost.py [--out FILE] [--k8-macro 20] [--reps 5]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

MODES = ("off", "es", "es_hist")


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, power, clk = [s.strip() for s in q.stdout.splitlines()[0].split(",")]
    return dict(gpu=name, power_limit=power, sm_clock_max=clk)


def alternate(run, set_mode, reps, stream):
    """run() is one timed replay; set_mode(m) switches statistics and histogram.  Returns per-mode lists of ms."""
    import torch
    res = {m: [] for m in MODES}
    for m in MODES:  # warm-up of every instantiation
        set_mode(m)
        run()
    torch.cuda.synchronize()
    for _ in range(reps):
        for m in MODES:
            set_mode(m)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            run(a, b)
            b.synchronize()
            res[m].append(a.elapsed_time(b))
    return res


def summary(res):
    med = {m: float(np.median(res[m])) for m in MODES}
    out = {f"ms_{m}": med[m] for m in MODES}
    out.update(ratio_es=med["es"] / med["off"], ratio_hist_vs_es=med["es_hist"] / med["es"],
               ratio_hist_vs_off=med["es_hist"] / med["off"])
    out.update({f"ms_{m}_all": res[m] for m in MODES})
    return out


def readback(b, stream, out):
    """One kfpos_batch_error_hist of all rows into a device tensor (events) and into host memory (wall clock)."""
    import torch
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    d = b.error_hist(readback=False, stream=stream)
    e1.record(stream)
    e1.synchronize()
    out["readback_device_ms"] = e0.elapsed_time(e1)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    h = b.error_hist(stream=stream)
    out["readback_host_ms"] = (time.perf_counter() - t0) * 1e3
    out["readback_bytes"] = int(h.nbytes)
    assert np.array_equal(d.cpu().numpy().astype(np.uint64), h)
    return h


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
    from roskfpos_b200.batch import Batch, epoch_summary, hist_quantiles

    if not torch.cuda.is_available():
        raise SystemExit("error_hist_cost.py: no CUDA device")
    dev = torch.device("cuda", 0)
    stream = torch.cuda.current_stream()
    out = dict(gpu_info(), reps=args.reps)
    N, T = args.filters, args.tsteps
    anc = synth.anchors_for(8)

    # ---- T6 headline, ERR histogram
    edges = np.arange(1, 201) * 0.01
    ranges, x0, _ = synth.device_ranges_mm(N, T, anc, 0.1, dev, seed=synth.SEED + 1000)
    truth = synth.device_truth_traj(N, T, 0.1, dev, seed=synth.SEED + 1000)
    x0f = torch.zeros((6, N), device=dev, dtype=torch.float64)
    x0f[:3] = x0
    with Batch(L.MODEL_T6, N, anchors=anc, accel_noise=0.5) as b:
        def set_mode(m):
            b.set_error_hist(edges if m == "es_hist" else None, "err")
            b.set_truth_traj(truth if m != "off" else None, stream=stream)

        def run(e0=None, e1=None):
            b.set_state(x0f, None, stream=stream)
            if e0 is not None:
                e0.record(stream)
            b.replay_toa(0.1, ranges, err=0.01, stream=stream)
            if e1 is not None:
                e1.record(stream)
        out["t6"] = summary(alternate(run, set_mode, args.reps, stream))
        out["t6"].update(filters=N, epochs=T, anchors=8, fmt="int32 mm, device resident", quantity="err",
                         n_edges=len(edges), edges="0.01 .. 2.00 m, 0.01 m steps",
                         kernel="t6_replay_kernel<false,false,8,false,1,ES,EH>")
        set_mode("es_hist")
        run()
        h = readback(b, stream, out["t6"])
        st = b.epoch_stats(stream=stream)
        out["t6"]["totals_match_epoch_stats"] = bool(np.array_equal(h.sum(axis=1), st[:, 2].astype(np.uint64)))
        lo, hi = hist_quantiles(h, edges, [0.5, 0.95])
        s = epoch_summary(st)
        out["t6"].update(rmse_last=float(s["rmse"][-1]), cep50_last=[float(lo[-1, 0]), float(hi[-1, 0])],
                         cep95_last=[float(lo[-1, 1]), float(hi[-1, 1])])
    del ranges, truth

    # ---- config-3 K8, NEES histogram
    nees_edges = np.concatenate([[0.0506, 0.103], np.arange(1, 101) * 0.25])  # chi2(2) 2.5 % / 5 %, then 0.25 steps
    w = synth.k8_montecarlo_chunk(N, 0, args.k8_macro, anc, dev, want_x0=True, want_truth_toa=True)
    with Batch(L.MODEL_K8, N, anchors=anc, xml=synth.K8_XML, accel_noise=0.5, jolt=0.5) as b:
        def set_mode(m):
            b.set_error_hist(nees_edges if m == "es_hist" else None, "nees")
            b.set_truth_traj(w["truth_toa"] if m != "off" else None, stream=stream)

        def run(e0=None, e1=None):
            b.set_state(w["x0"], None, stream=stream)
            if e0 is not None:
                e0.record(stream)
            b.replay_events(w["events"], ranges=w["ranges"], sensors=w["sensors"], err=0.01, stream=stream)
            if e1 is not None:
                e1.record(stream)
        out["config3_k8"] = summary(alternate(run, set_mode, args.reps, stream))
        out["config3_k8"].update(filters=N, macro_steps=args.k8_macro, events=w["n_events"], toa_rows=w["n_toa"],
                                 quantity="nees", n_edges=len(nees_edges),
                                 kernel="k8_replay_kernel<false,8,false,false,ES,EH>")
        set_mode("es_hist")
        run()
        h = readback(b, stream, out["config3_k8"])
        st = b.epoch_stats(stream=stream)
        out["config3_k8"]["totals_match_epoch_stats"] = bool(np.array_equal(h.sum(axis=1),
                                                                            st[:, 5].astype(np.uint64)))
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
