"""Cost of the per-epoch Cramer-Rao bound (kfpos_batch_crlb) and what it shows.

Timed with CUDA events around the calls only, sets alternated within each repetition (median of --reps):
  kernel     1 Mi filters x 1000 epochs x 8 anchors, int32, p_missing = p_nlos = 0.05: the bound of each set
             (PRESENT, LOS, USED with the variant-1 selection of a T6 replay of the log) with the scalar variance;
             ms, bytes read per second (n_rows N (M 4 + 24 [+ 4 mask] [+ 4 sel])) next to a device-to-device
             cudaMemcpyAsync of the log, the truth, the mask and `sel` timed in the same run, and the FP64 rate
             next to the DFMA peak of kfpos_measure_fp64_peak; the ptxas registers and spills of the kernels
  accuracy   8 anchors, 64 Ki filters x 1000 epochs, sigma_r 0.10 m with errorEstimation 0.10 m, 5 % NLOS of mean
             0.8 m (DESIGN §4.5c / §4.5d): final RMSE, the mean over the epochs of the PRESENT, LOS and USED RMS
             floors (batch.crlb_summary) and the final RMSE over the final USED floor, for T6 none / leave-one-out
             / variant 1 / variant 2 (synth.toa_montecarlo(crlb=...)) and ML variant 1 (n = 1) / variant 2, epoch
             by epoch
Prints one JSON object with the GPU's name, power limit and max SM clock.

    python profiles/crlb_cost.py [--out FILE] [--reps 5]
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import re
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from epoch_stats_cost import gpu_info  # noqa: E402
from synth_toa_cost import alternate  # noqa: E402

HBM_BYTES_PER_S = 7.7e12  # NVIDIA HGX B200 data sheet, one GPU
SETS = ("present", "los", "used")
# FP64 operations per (filter, row) at 8 anchors: per anchor 3 differences, a 3-term square sum, the reciprocal
# square root (5), 3 products for g, 3 weighted components and 6 information sums (~23); the LDL^T and the
# trace with its 6 divisions (~60): the issue's estimate of ~250, kept as an order of magnitude
FP64_OPS_PER_ROW = 250


def ptxas_counts():
    """Registers and spill bytes of every crlb_kernel instantiation, from the build's ptxas log."""
    path = os.path.join(ROOT, "roskfpos_b200", "csrc", "kfpos_crlb.ptxas.log")
    if not os.path.exists(path):
        return None
    out, name = {}, None
    for line in open(path):
        m = re.search(r"Function properties for (\S*crlb_kernel\S*)", line)
        if m:
            name = re.search(r"crlb_kernelILi(\d)ELi(\d)", m.group(1)).groups()
            name = "crlb_kernel<fmt %s, D %s>" % name
            continue
        m = re.search(r"(\d+) bytes spill stores, (\d+) bytes spill loads", line)
        if m and name:
            out.setdefault(name, {})["spill_bytes"] = int(m.group(1)) + int(m.group(2))
        m = re.search(r"Used (\d+) registers", line)
        if m and name:
            out.setdefault(name, {})["registers"] = int(m.group(1))
            name = None
    return out


def floors(rows):
    from roskfpos_b200.batch import crlb_summary
    s = crlb_summary(rows)
    return float(np.nanmean(s["rmse_bound"])), float(s["rmse_bound"][-1])


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
    from roskfpos_b200.batch import Batch, epoch_summary

    if not torch.cuda.is_available():
        raise SystemExit("crlb_cost.py: no CUDA device")
    dev = torch.device("cuda", 0)
    stream = torch.cuda.current_stream()
    out = dict(gpu_info(), reps=args.reps, ptxas=ptxas_counts())
    N, T, M = args.filters, args.epochs, 8
    anc = synth.anchors_for(M)
    imp = dict(p_missing=0.05, p_nlos=0.05, nlos_mean=0.8, sigma_r=0.10)
    var = 0.10 ** 2 + 1e-6 / 12

    # ---- (a) the kernel on the headline shape, next to a copy of its inputs
    w = synth.toa_montecarlo_chunk(N, 0, T, anc, dev, stream=stream, want_nlos=True, want_x0=True, want_truth=True,
                                   **imp)
    sel = torch.empty((T, N), dtype=torch.int32, device=dev)
    rows = {s: torch.empty((T, L.CRLB_COLS), dtype=torch.float64, device=dev) for s in SETS}
    with Batch(L.MODEL_T6, N, anchors=anc, accel_noise=0.5, variant=1, num_ignored_rangings=1) as b:
        b.set_state(w["x0"], None, stream=stream)
        b.replay_toa(w["dt"], w["ranges"], err=0.10, sel=sel, stream=stream)
        call = lambda s: lambda: b.crlb(w["truth"], w["ranges"], var, sel, w["nlos"], set=s, out=rows[s],
                                        stream=stream)
        src = [w["ranges"], w["truth"], w["nlos"], sel]
        dst = [torch.empty_like(x) for x in src]

        def copy():
            for d, s in zip(dst, src):
                d.copy_(s)
        res = alternate({**{s: call(s) for s in SETS}, "copy": copy}, args.reps, stream)
        summary = {s: dict(zip(("mean_floor_m", "final_floor_m"), floors(rows[s].cpu().numpy()))) for s in SETS}
    del dst
    torch.cuda.empty_cache()
    peak = C.c_double(0.0)
    L.check(L.lib().kfpos_measure_fp64_peak(0, C.byref(peak)), "kfpos_measure_fp64_peak")
    base = T * N * (M * 4 + 24)
    nbytes = dict(present=base, los=base + 4 * T * N, used=base + 4 * T * N)
    copy_bytes = sum(x.numel() * x.element_size() for x in src)
    cp = float(np.median(res["copy"]))
    copy_rate = copy_bytes / (cp * 1e-3)
    cases = {}
    for s in SETS:
        ms = float(np.median(res[s]))
        rate = nbytes[s] / (ms * 1e-3)
        fp64 = FP64_OPS_PER_ROW * T * N / (ms * 1e-3)
        cases[s] = dict(ms=ms, ms_all=res[s], bytes_read=nbytes[s], read_gb_per_s=rate / 1e9,
                        read_share_of_hbm_datasheet=rate / HBM_BYTES_PER_S, read_over_copy_rate=rate / copy_rate,
                        datasheet_bound_ms=nbytes[s] / HBM_BYTES_PER_S * 1e3, fp64_ops_per_s_est=fp64,
                        fp64_share_of_measured_peak_est=fp64 / peak.value, **summary[s])
    out["kernel"] = dict(filters=N, rows=T, anchors=M, fmt="int32", impaired=imp, var=var,
                         selection="T6 variant 1 (n = 1)", cases=cases, copy_ms=cp, copy_ms_all=res["copy"],
                         copy_bytes=copy_bytes, copy_gb_per_s=copy_bytes / cp / 1e6,
                         fp64_peak_flops_measured=peak.value, fp64_ops_per_row_est=FP64_OPS_PER_ROW,
                         note="copy_gb_per_s counts each copied byte once; the copy reads and writes it; the FP64 "
                              "rate counts FP64_OPS_PER_ROW operations per (filter, row), an estimate, not a count")
    del w, sel, src, rows
    torch.cuda.empty_cache()

    # ---- (b) the accuracy table of DESIGN §4.5d with the floors, 64 Ki filters x 1000 epochs
    NA = args.acc_filters
    acc = {}
    kw = dict(p_nlos=0.05, nlos_mean=0.8, sigma_r=0.10)
    t6_modes = {"t6_none": {}, "t6_leave_one_out": dict(ignore_worst_anchor=1),
                "t6_variant1_n1": dict(variant=1, num_ignored_rangings=1), "t6_variant2": dict(variant=2)}

    def row(final_rmse, cr):
        f = {s: floors(cr[s]) for s in SETS}
        return dict(final_rmse=final_rmse, **{"mean_floor_" + s: f[s][0] for s in SETS},
                    **{"final_floor_" + s: f[s][1] for s in SETS}, final_rmse_over_used_floor=final_rmse / f["used"][1])
    for name, cfg in t6_modes.items():
        with Batch(L.MODEL_T6, NA, anchors=anc, accel_noise=0.5, **cfg) as b:
            rows_, cr = synth.toa_montecarlo(b, T, T, anc, err=0.10, stream=stream, crlb=SETS, **kw)
        acc[name] = row(float(epoch_summary(rows_)["rmse"][-1]), cr)
    for name, cfg in (("ml_variant1_n1", dict(variant=1, num_ignored_rangings=1)), ("ml_variant2", dict(variant=2))):
        ch = {}
        with Batch(L.MODEL_ML, NA, anchors=anc, **cfg) as b:
            o = dict(pos=torch.empty((3, NA), dtype=torch.float64, device=dev),
                     sel=torch.empty((2, NA), dtype=torch.int32, device=dev),
                     status=torch.empty(NA, dtype=torch.int32, device=dev))
            cr = {s: torch.empty((T, L.CRLB_COLS), dtype=torch.float64, device=dev) for s in SETS}
            wc = synth.toa_montecarlo_chunk(NA, 0, T, anc, dev, out=ch, want_truth=True, want_nlos=True,
                                            stream=stream, **kw)
            for k in range(T):
                b.ml_solve(wc["ranges"][k], err=0.10, out=o, stream=stream)
                for s in SETS:
                    b.crlb(wc["truth"][k], wc["ranges"][k], var, o["sel"], wc["nlos"][k], set=s,
                           out=cr[s][k:k + 1], stream=stream)
            e2 = ((o["pos"] - wc["truth"][-1]) ** 2).sum(dim=0)
            e2 = e2[torch.isfinite(e2)]
            acc[name] = row(float(torch.sqrt(e2.mean())), {s: cr[s].cpu().numpy() for s in SETS})
    out["accuracy"] = dict(filters=NA, epochs=T, anchors=M, err=0.10, var=var, modes=acc,
                           ml_note="ML batches solve each epoch alone from ml_start (1, 1, 4); final RMSE = the last "
                                   "epoch's estimates against its truth", **kw)
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
