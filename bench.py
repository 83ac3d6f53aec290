#!/usr/bin/env python
"""bench.py -- EKF filter-updates/s @ 8 anchors (BASELINE.json metric).

One bench "step" = one pass of the hot path over one batch: reset N filters to
their initial positions, replay T ranging epochs through the persistent IEKF
kernel (KalmanFilterTOA, 8 anchors, int32-mm SoA range log resident in HBM),
reduce the error statistics.  value = N_total * T * K / elapsed.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference]
  torchrun --nproc-per-node N bench.py --gpus N ...      (one rank per GPU)

Prints ONE JSON line (rank 0).  See DESIGN.md "Measurement" for every field.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "ekf_filter_updates_per_sec_8anchors"
UNIT = "updates/s"


def w_alg_t6(m, i_ml, i_c, i_g):
    """Algorithmic FLOP per T6 update, SURVEY.md §8(d) formula W_alg (v1); the
    iteration counts are the MEASURED per-update means from the device counters."""
    w_pred = 4 * 3 * 6 + 12 + 15 + 2 * 3
    w_mlit = 59 * m + 60
    w_cost = 13 * m + (2 * 3 * m + 3 * m) + 3
    w_gain = (1 + 3) * m + m * (36 + 2 * 6 * 3 + 4 * 6 + 4 * 3 + 3) + 6
    return w_pred + i_ml * w_mlit + 12 * m + 2 * m + i_c * w_cost + i_g * w_gain


def w_alg_t6_v2(m, i_ml, i_c, i_g):
    """Algorithmic FLOP per T6 update of the formulation the kernel actually uses (information-form IEKF, one pass
    per Newton / IEKF iteration, first pass shared, factored covariance update); DESIGN.md §4.0 "W_alg v2".  Same
    conventions as SURVEY.md §8(d): add / mul / rsqrt / rcp = 1, FMA = 2."""
    w_pred = 105
    pass_ml = 37 * m + 60          # distances, residual, gradient, 5 of 6 Hessian sums, 3x3 solve, stop test
    pass_first = 49 * m + 60       # + the 5 sums of u u^T that the first IEKF iteration reuses
    pass_iekf = 32 * m + 20        # cost, b, 5 of 6 sums of G, G dx
    gain = 184                     # N = I + G A, cofactors, s, dx, M, prior, scaling by 1/R
    apply = 216                    # P^- - B M B^T on the packed 6x6
    return w_pred + 2 * m + pass_first + i_ml * pass_ml + (i_c - 1) * pass_iekf + 5 * i_c + i_g * gain + apply


K8_ROWS = {"px4": ((4, 4, 1), 24), "imu": ((3, 3, 1), 7), "mag": ((1,), 1)}  # nnz per row, c_q (SURVEY.md §8d)


def w_alg_k8(m, sensors, i_ml, i_c, i_g):
    """Algorithmic FLOP of one K8 event, SURVEY.md §8(d) formula W_alg (v1) for n = 8, d = 2: m valid rangings
    (0 for a sensor-only event) fused with the sensor groups in `sensors`; the iteration counts are MEASURED means.
    (Nominal counts reproduce the table of §8d: 1994 PX4-only, 726 mag-only, 8003 TOA + IMU + mag, 1790 IMU-only.)"""
    n, d = 8, 2
    rows = [d] * m + [z for s_ in sensors for z in K8_ROWS[s_][0]]
    q = len(rows) - m
    nnz_q = sum(rows[m:])
    c_q = sum(K8_ROWS[s_][1] for s_ in sensors)
    w_pred = 4 * 7 * n + 22 + 15 + 2 * 7
    w_ml = (12 * m + i_ml * (46 * m + 25) + 12 * m) if m > 0 else 0.0
    w_cost = 13 * m + q + c_q + (2 * d * m + 2 * nnz_q + 3 * len(rows)) + 3
    w_gain = (1 + d) * m + (10 if q > 0 else 0) + sum(n * n + 2 * n * z + 4 * n + 4 * z + 3 for z in rows) + n
    return w_pred + w_ml + 2 * m + (6 if len(rows) >= 3 else 0) + i_c * w_cost + i_g * w_gain


def k8_roofline(events, full, m, N, cnt, seconds, peak):
    """FP64 roofline block of a K8 replay: sum of W_alg over the schedule (what each event fuses follows from the
    schedule: every sensor is latched by the first macro-step) with the measured mean iteration counts."""
    from roskfpos_b200 import synth
    n_upd = max(cnt["updates"], 1.0)
    n_toa = sum(1 for e in events if e[0] == synth.EV_TOA)
    i_c, i_g = cnt["cost_evals"] / n_upd, cnt["gain_evals"] / n_upd
    i_ml = cnt["ml_iters"] / max(N * n_toa, 1)
    latched = ("px4", "imu", "mag") if full else ("imu", "mag")
    fused = {synth.EV_IMU: (0, ("imu",)), synth.EV_PX4: (0, ("px4",)), synth.EV_MAG: (0, ("mag",)),
             synth.EV_COMPASS: (0, latched), synth.EV_TOA: (m, latched)}
    w = sum(w_alg_k8(fused[e[0]][0], fused[e[0]][1], i_ml, i_c, i_g) for e in events)
    ach = w * N / seconds
    return {"bound": "fp64", "achieved": ach / 1e12, "peak": peak / 1e12, "unit": "TFLOP/s",
            "frac": ach / peak if peak else None, "flop_per_event_mean": w / len(events),
            "mean_iters": {"ml_per_toa": i_ml, "cost": i_c, "gain": i_g}, "kernel": "k8_replay_kernel<false,8,false>",
            "numerator": "SURVEY.md §8(d) W_alg v1 per event kind (IMU 3 rows, PX4 3 rows, compass = mag + latched "
                         "sensors, TOA = 8 rangings + latched sensors) with the measured iteration counters",
            "peak_source": "measured live: kfpos_measure_fp64_peak"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50",
                 "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thr = threading.Thread(target=self._read, daemon=True)
            self.thr.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), [c.strip() for c in line.split(",")]))

    def window(self, t0, t1):
        """keep only the samples that arrived inside the timed region [t0, t1]"""
        self.t0, self.t1 = t0, t1

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, smax, reasons, pw = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        t0, t1 = getattr(self, "t0", None), getattr(self, "t1", None)
        rows = [r for (ts, r) in self.rows if t0 is None or (t0 <= ts <= t1 + 0.05)]
        if not rows:  # timed region shorter than the sampling period: nearest samples
            rows = [r for (_, r) in self.rows[-3:]]
        for r in rows:
            try:
                sm.append(float(r[1])); smax.append(float(r[2])); pw.append(float(r[3]))
            except (ValueError, IndexError):
                continue
            for n, v in zip(names, r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None,
                "sm_max_mhz": max(smax) if smax else None,
                "power_w_max": max(pw) if pw else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def load_t6_counters():
    """ncu counters of ONE launch of the headline kernel, committed under profiles/ (per update, so that they
    scale to any batch size): executed FP64 instruction mix and DRAM bytes.  profiles/r02_t6_counters.json is
    written by profiles/extract_counters.py from the .ncu-rep of the same bench command."""
    p = os.path.join(ROOT, "profiles", "r02_t6_counters.json")
    if os.path.exists(p):
        return json.load(open(p))
    return None


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return json.load(open(p)), "measured"
    return {"hbm_gbs": 6650.0}, "fallback"


# --------------------------------------------------------------------------- CPU
def _ref_worker(job):
    """One single-threaded reference process (the reference is single-threaded,
    node_pos.cpp:176-181): generates its slice, times only the filter calls."""
    seed, nf, tsteps, n_anchors = job
    from oracle import ref_py as R
    from roskfpos_b200 import synth
    anc = synth.anchors_for(n_anchors)
    truth = synth.truth_lissajous(nf, tsteps, 0.1, seed=seed)
    r = synth.ranges_mm(truth[1:], anc, seed=seed + 1).astype(np.float64) / 1000
    R.lib()
    t0 = time.perf_counter()
    out = R.t6_replay(truth[0], r, anc, 0.1, 0.01)
    return time.perf_counter() - t0, nf * tsteps, int(out["rc"])


def cpu_reference(n_anchors, tsteps, seconds, threads=0):
    """Times the reference's CPU implementation of the path on a bounded sample of the bench
    workload, on all host cores.  kind "reference": the reference's own .cpp files compiled
    against the shim headers + LAPACK (oracle/_ref, one process per core); kind "port": the
    oracle restatement with OpenMP (when oracle/_ref was not built)."""
    from oracle import oracle_py as O
    from oracle import ref_py as R
    from roskfpos_b200 import synth
    anc = synth.anchors_for(n_anchors)
    cores = threads or os.cpu_count() or 1
    if R.available():
        import multiprocessing as mp
        ctx = mp.get_context("fork")
        with ctx.Pool(cores) as pool:
            probe = pool.map(_ref_worker, [(synth.SEED + 50 + i, 8, tsteps, n_anchors) for i in range(cores)])
            rate_core = np.mean([u / t for t, u, _ in probe])
            nf = int(max(8, rate_core * seconds / tsteps))
            res = pool.map(_ref_worker, [(synth.SEED + 100 + i, nf, tsteps, n_anchors) for i in range(cores)])
        tt = max(t for t, _, _ in res)
        upd = sum(u for _, u, _ in res)
        # the reference's native mode (SURVEY.md §8d-i): ONE filter, one thread, BASELINE config 1 (4 anchors,
        # 10 000 steps at 10 Hz)
        t1, u1, _ = _ref_worker((synth.SEED + 1, 1, 10000, 4))
        native = {"updates_per_s": u1 / t1, "us_per_update": 1e6 * t1 / u1,
                  "sample": "1 filter x 10000 steps, 4 anchors (BASELINE config 1a), one thread"}
        return {"value": upd / tt, "unit": UNIT, "cores": cores, "kind": "reference", "single_filter": native,
                "sample": f"{nf * cores} filters x {tsteps} steps, {n_anchors} anchors, the reference's own "
                          f"KalmanFilterTOA.cpp + MLLocation.cpp (g++ -O2, shim Armadillo over OpenBLAS LAPACK), "
                          f"{cores} single-threaded processes, {tt:.1f} s",
                "errors": int(sum(rc for _, _, rc in res))}

    def run(nf):
        truth = synth.truth_lissajous(nf, tsteps, 0.1, seed=synth.SEED + 7)
        r = synth.ranges_mm(truth[1:], anc, seed=synth.SEED + 8)
        t0 = time.perf_counter()
        out = O.t6_replay(truth[0], None, r, anc, 0.1, 0.01, threads=cores)
        return time.perf_counter() - t0, out

    cores = threads or O.max_threads()
    probe_n = 64 * cores
    tp, _ = run(probe_n)
    rate = probe_n * tsteps / max(tp, 1e-6)
    nf = int(max(probe_n, min(rate * seconds / tsteps, 4_000_000)))
    tt, out = run(nf)
    upd = nf * tsteps
    return {"value": upd / tt, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"{nf} filters x {tsteps} steps, {n_anchors} anchors, T6 (KalmanFilterTOA) oracle "
                      f"restatement, gcc -O3 + OpenMP, {tt:.1f} s",
            "mean_iters": {"ml": out["counters"][0] / upd, "cost": out["counters"][1] / upd,
                           "gain": out["counters"][2] / upd}}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    K, W = args.steps, args.warmup
    per = max(2.0, min(20.0, 100.0 / max(K + W, 1)))
    vals = []
    last = None
    t_steps = []
    for i in range(W + K):
        t0 = time.perf_counter()
        last = cpu_reference(args.anchors, args.tsteps, per)
        if i >= W:
            vals.append(last["value"])
            t_steps.append(time.perf_counter() - t0)
    v = float(np.mean(vals))
    last["value"] = v
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus,
            "steps": K, "warmup": W, "ms_per_step": 1e3 * float(np.mean(t_steps)), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": f"T6 (KalmanFilterTOA) IEKF replay, {args.anchors} anchors, dt 0.1 s, P0=0, fixed "
                                   f"initial position; bounded CPU sample per step (see cpu_baseline.sample)",
                       "anchors": args.anchors, "epochs_per_step": args.tsteps},
            "cpu_baseline": last,
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# --------------------------------------------------------------------------- GPU
def run_b200(args):
    import torch
    import torch.distributed as dist
    from roskfpos_b200 import lib as L, synth
    from roskfpos_b200.batch import Batch
    from roskfpos_b200.shard import reduce_stats

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product has no CPU path "
                         "(use --impl reference for the CPU baseline)")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        # keep stdout to the single JSON line: NCCL prints its version banner there at VERSION level
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ["NCCL_DEBUG"] = "WARN"
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    N, T, M, K, W = args.filters, args.tsteps, args.anchors, args.steps, args.warmup

    anc = synth.anchors_for(M)
    ranges, x0, truth_end = synth.device_ranges_mm(N, T, anc, 0.1, dev, seed=synth.SEED + 1000 * rank)
    x0_full = torch.zeros((6, N), device=dev, dtype=torch.float64)
    x0_full[:3] = x0
    batch = Batch(L.MODEL_T6, N, device=local, anchors=anc, accel_noise=0.5)
    stream = torch.cuda.current_stream()
    # the ground truth is registered once: every replay launch then ends with the block-level reduction of the
    # error statistics, a step only adds the final tree (no host synchronisation inside the timed loop)
    batch.set_truth(truth_end, stream=stream)
    # the job's one collective goes through the C ABI (kfpos_stats_allreduce) on a raw NCCL communicator
    comm = None
    if world > 1:
        from roskfpos_b200.shard import nccl_comm
        comm = nccl_comm(rank, world, local)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step_resident():
        batch.set_state(x0_full, None, stream=stream)
        batch.replay_toa(0.1, ranges, err=0.01, stream=stream)
        batch.error_stats(stream=stream, readback=False)

    # ---- device-resident throughput (`value`)
    sampler = ClockSampler(local)
    sampler.start()  # every rank watches its own GPU
    for _ in range(W):
        step_resident()
    # the warm-up includes the job's collective: the first call on a fresh NCCL communicator sets up its
    # connections (6-140 ms from box to box), which is not part of a step
    batch.stats_allreduce(comm, stream=stream)
    batch.counters(reset=True)
    barrier()
    t_start = time.perf_counter()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    kev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    torch.cuda.cudart().cudaProfilerStart()  # ncu --profile-from-start off sees the timed region only
    e0.record(stream)
    for k in range(K):
        batch.set_state(x0_full, None, stream=stream)
        kev[k][0].record(stream)
        batch.replay_toa(0.1, ranges, err=0.01, stream=stream)
        kev[k][1].record(stream)
        batch.error_stats(stream=stream, readback=False)  # the final tree over the block partials; stays on the device
    # the only collective of the job: the final reduction of the statistics (filters are independent,
    # so nothing forces the ranks into lock-step between the steps); one ncclAllGather of 4 doubles + D2H
    s = batch.stats_allreduce(comm, stream=stream)
    e1.record(stream)
    barrier()
    torch.cuda.cudart().cudaProfilerStop()
    sampler.window(t_start, time.perf_counter())
    clocks = sampler.stop()
    ms = e0.elapsed_time(e1)
    kernel_ms = float(np.mean([a.elapsed_time(b) for a, b in kev]))
    per_rank = [{"rank": rank, "kernel_ms": kernel_ms, "sm_mhz": clocks.get("sm_mhz"),
                 "power_w_max": clocks.get("power_w_max"), "reasons": clocks.get("reasons")}]
    if world > 1:
        gathered = [None] * world
        dist.all_gather_object(gathered, per_rank[0])
        per_rank = gathered
    cnt = batch.counters(reset=True)
    t = torch.tensor([ms], device=dev, dtype=torch.float64)
    rank_ms = [ms]
    if world > 1:
        allt = [torch.zeros_like(t) for _ in range(world)]
        dist.all_gather(allt, t)
        rank_ms = [float(v.item()) for v in allt]
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max = float(t.item())
    value = world * N * T * K / (ms_max * 1e-3)
    rmse = float(s[4])
    if args.dump_outputs and rank == 0:  # before the e2e leg replays other epochs on the same batch
        dump_outputs(args.dump_outputs, batch, s, stream)

    # ---- end to end through the C ABI with HOST (pinned) buffers
    e2e = None
    if not args.no_e2e:
        # the host log holds the first Te epochs of the same workload (pinned host memory is bounded: 1000
        # epochs would be 33.5 GB per rank); the per-update rate is what is compared
        import ctypes as C
        Te = min(T, args.e2e_tsteps)
        h_x0 = torch.empty(x0_full.shape, dtype=torch.float64, pin_memory=True)
        h_x0.copy_(x0_full)
        h_truth = torch.empty(truth_end.shape, dtype=torch.float64, pin_memory=True)
        h_truth.copy_(truth_end)
        h_pos = torch.empty((6, N), dtype=torch.float64, pin_memory=True)
        hx, ht, hp = h_x0.numpy(), h_truth.numpy(), h_pos.numpy()
        Ke = max(1, min(K, 3))

        def e2e_leg(h_log):
            hr = h_log.numpy()

            def step_e2e():
                batch.set_state(hx, None, stream=stream)                      # H2D x0
                batch.replay_toa(0.1, hr, err=0.01, stream=stream)            # H2D range log, chunked + overlapped
                s_ = batch.error_stats(ht, stream=stream)                     # H2D truth, D2H 4 doubles
                L.check(L.lib().kfpos_batch_get_state(batch._h, C.c_void_p(hp.ctypes.data), None, None,
                                                      C.c_void_p(stream.cuda_stream)), "get_state")  # D2H x
                return s_
            for _ in range(max(1, min(W, 2))):
                step_e2e()
            barrier()
            t0 = time.perf_counter()
            f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            f0.record(stream)
            for _ in range(Ke):
                s_last = step_e2e()
            f1.record(stream)
            barrier()
            wall = (time.perf_counter() - t0) * 1e3
            ems = max(f0.elapsed_time(f1), 0.0)
            te = torch.tensor([max(ems, wall if world == 1 else ems)], device=dev, dtype=torch.float64)
            if world > 1:
                dist.all_reduce(te, op=dist.ReduceOp.MAX)
            h2d = int(h_log.numel() * h_log.element_size() + 8 * 6 * N + 8 * 3 * N)
            ms_e = float(te.item())
            return {"value": world * N * Te * Ke / (ms_e * 1e-3), "unit": UNIT, "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": int(8 * 6 * N + 32), "steps": Ke, "epochs_per_step": Te,
                    "ms_per_step": ms_e / Ke, "h2d_gbs": h2d * Ke / (ms_e * 1e-3) / 1e9}, s_last

        # the library's wire format for host-resident range logs: uint16 millimetres (every UWB range is < 65.5 m);
        # the step is bound by the host-to-device copy, and the box's PCIe / host memory gives what it gives
        # (profiles/r02_h2d_ngpu.txt: 55.5 GB/s per GPU alone, 23-36 GB/s with 8 GPUs copying), so the width of
        # the wire format is the one lever -- the kernel converts either format to metres bit-identically
        h16 = torch.empty((Te,) + tuple(ranges.shape[1:]), dtype=torch.uint16, pin_memory=True)
        h16.copy_(ranges[:Te].to(torch.uint16))
        e2e, s16 = e2e_leg(h16)
        e2e["wire_format"] = "uint16 mm (KFPOS_FMT_U16_MM)"
        e2e["note"] = ("host range log in the library's uint16-mm wire format; the step is bound by the host-to-device "
                       "copy (h2d_gbs), which the replay kernel overlaps chunk by chunk; int32_table_format = the same "
                       "step with the log in the reference's int32-mm table format (PG.cpp:213)")
        del h16
        try:
            h32 = torch.empty((Te,) + tuple(ranges.shape[1:]), dtype=ranges.dtype, pin_memory=True)
            h32.copy_(ranges[:Te])
            leg32, s32 = e2e_leg(h32)
            leg32["rmse_equal"] = bool(abs(s32[0] - s16[0]) <= 1e-12 * abs(s16[0]))
            e2e["int32_table_format"] = leg32
            del h32
        except Exception as exc:  # an extra, never fatal
            e2e["int32_table_format"] = {"error": repr(exc)}

    # ---- roofline of the dominant kernel (t6_replay_kernel): FP64 CUDA-core bound
    upd = max(cnt["updates"], 1.0)
    i_ml, i_c, i_g = cnt["ml_iters"] / upd, cnt["cost_evals"] / upd, cnt["gain_evals"] / upd
    w_alg = w_alg_t6(M, i_ml, i_c, i_g)
    peak = C_double_peak(local)
    ach = w_alg * N * T / (kernel_ms * 1e-3)
    peaks, peak_src = load_peaks()
    alg_bytes = N * T * M * ranges.element_size() + N * (3 + 21) * 8 * 2
    # executed work and DRAM traffic of ONE launch, from the committed ncu capture of this kernel (per update)
    ctr = load_t6_counters() if M == 8 else None
    traffic = frac_exec = exec_flop = None
    if ctr:
        traffic = ctr["dram_bytes_per_update"] * N * T
        exec_flop = ctr["executed_flop_per_update"]
        frac_exec = exec_flop * N * T / (kernel_ms * 1e-3) / peak if peak else None
    roof = {"bound": "fp64", "achieved": ach / 1e12, "peak": peak / 1e12, "unit": "TFLOP/s",
            "frac": ach / peak if peak else None, "traffic": traffic, "traffic_unit": "bytes per launch",
            "traffic_source": ctr and ctr.get("source"),
            "frac_executed": frac_exec, "executed_flop_per_update": exec_flop,
            "executed_note": "2*DFMA + DMUL + DADD thread instructions (smsp__sass_thread_inst_executed_op_d*_pred_on) "
                             "of the committed ncu capture / updates of that launch, times this run's update rate",
            "algorithmic_bytes": alg_bytes,
            "peak_source": "measured live: kfpos_measure_fp64_peak (DFMA-only kernel, best of 5)",
            "kernel": "t6_replay_kernel<PME=0,LOO=0,MT=8,SEL=0,FMT=1 (int32 mm)>", "kernel_ms": kernel_ms,
            "flop_per_update": w_alg, "mean_iters": {"ml": i_ml, "cost": i_c, "gain": i_g},
            "flop_per_update_v2": w_alg_t6_v2(M, i_ml, i_c, i_g),
            "frac_v2": w_alg_t6_v2(M, i_ml, i_c, i_g) * N * T / (kernel_ms * 1e-3) / peak if peak else None,
            "v2_note": "W_alg v2 = the algorithmic count of the information-form formulation the kernel uses (DESIGN.md "
                       "§4.0); frac >= frac_executed >= frac_v2 bracket the useful share of the FP64 peak",
            "numerator": "SURVEY.md §8(d) W_alg v1 (sequential-scalar IEKF count) with the measured iteration "
                         "counters; the kernel's information-form IEKF executes fewer flops than that count "
                         "(profiles/README.md: executed FP64 instructions per update from ncu)",
            "hbm": {"achieved_gbs": alg_bytes / (kernel_ms * 1e-3) / 1e9, "peak_gbs": peaks.get("hbm_gbs"),
                    "peak_source": peak_src, "bytes_per_update": alg_bytes / (N * T)}}

    # ---- BASELINE config 5 (64 Mi K8 filters in TOTAL over the ranks: strong scaling), every world size
    del ranges
    torch.cuda.empty_cache()
    config5 = None
    if not args.no_config5:
        try:
            config5 = config5_leg(local, dev, world, rank, comm, args.config5_filters, 2, 2, 1, full=True)
        except Exception as exc:  # a secondary number must never take the headline line down
            config5 = {"error": repr(exc)}
            if world > 1:
                raise
    other = None
    if rank == 0 and world == 1 and not args.no_extra:
        try:
            other = bench_other_configs(local, dev, args)
        except Exception as exc:  # secondary numbers must never take the headline line down
            other = {"error": repr(exc)}
    if rank == 0:
        cpu = None if args.no_cpu else cpu_reference(M, min(T, 100), args.cpu_seconds)
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
                "ms_per_step": ms_max / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f64", "data": "synthetic",
                "config": {"workload": f"T6 (KalmanFilterTOA) IEKF replay: {N} filters/GPU x {T} epochs, "
                                       f"{M} anchors, int32-mm ranges, dt 0.1 s, P0=0, fixed initial position",
                           "filters_per_gpu": N, "epochs_per_step": T, "anchors": M,
                           "l2_policy": f"inputs larger than L2 ({N * T * M * 4 / 1e6:.0f} MB range log per step)",
                           "parallelism": f"filters sharded by index over {world} GPU(s); one all-reduce of 4 doubles at the end"},
                "rmse_m": rmse, "bad_updates": cnt["bad"], "rank_ms_per_step": [v / K for v in rank_ms], "ranks": per_rank,
                "e2e": e2e, "gpu_launches": 2 * K + 1 + (1 if world > 1 else 0), "roofline": roof, "cpu_baseline": cpu,
                "clocks": clocks, "timed_region_s": ms_max * 1e-3,
                "config5": config5, "other_configs": other}
        print(json.dumps(line))
    batch.close()
    if comm is not None:
        comm.close()
    if world > 1:
        dist.destroy_process_group()


def dump_outputs(out_dir, batch, stats, stream, n_sample=1 << 16):
    """What the last timed step hands its caller, as float64 .npy files under `out_dir`: the state `x` [n][S],
    covariance `P` [n*n][S] and status words `status` [S] of a fixed sample of S <= n_sample filters (their
    indices in `filter_index`; every filter when N <= n_sample) and the reduced statistics `error_stats` [6].
    The sample depends on N alone, so two builds run with the same arguments can be compared file by file.
    It is gathered on the device, so the host holds the dump alone: 8 (n*n + n + 2) bytes per sampled filter,
    23 MB for T6 (n = 6), 39 MB for K8 (n = 8).  A directory created here ignores itself in git."""
    import torch
    from roskfpos_b200 import synth
    N, n = batch.N, batch.n
    dev = torch.device("cuda", torch.cuda.current_device())
    idx = np.arange(N) if N <= n_sample else np.sort(np.random.default_rng(synth.SEED).choice(N, n_sample, replace=False))
    sel = torch.as_tensor(idx, device=dev)
    out = {"filter_index": idx, "error_stats": stats}
    for name, shape, dtype in (("x", (n, N), torch.float64), ("P", (n * n, N), torch.float64),
                               ("status", (N,), torch.int32)):
        full = torch.empty(shape, device=dev, dtype=dtype)
        batch.get_state_into(**{name: full}, stream=stream)
        out[name] = full.index_select(-1, sel).cpu().numpy()
        del full
    if not os.path.isdir(out_dir):
        os.makedirs(out_dir)
        with open(os.path.join(out_dir, ".gitignore"), "w") as f:
            f.write("*\n")
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a, dtype=np.float64))


def config5_leg(local, dev, world, rank, comm, total_filters, n_macro, K, W, full=True, chunk=None, dump=None):
    """BASELINE config 5 (full=False: config 3) as a STRONG-scaling leg: `total_filters` K8 filters in total,
    sharded by index over the ranks, inputs generated on the device chunk by chunk inside the timed region
    (never resident), statistics fused into the replay, ONE collective at the end (kfpos_stats_allreduce).
    Generator and summation tree depend on the global filter index only, so the reduced statistics are
    bit-identical for any number of GPUs: the hex strings of the returned dict are there to be compared.
    dump: a directory for dump_outputs of this rank's batch after the timed steps."""
    import torch
    import torch.distributed as dist
    from roskfpos_b200 import lib as L, synth
    from roskfpos_b200.batch import Batch
    from roskfpos_b200.shard import shard_bounds
    stream = torch.cuda.current_stream()
    macro = synth.MACRO_FULL if full else synth.MACRO_IMU_MAG
    lo, hi = shard_bounds(total_filters, rank, world)
    N = hi - lo
    if chunk is None:
        chunk = 2 if full else max(1, min(n_macro, (3 << 30) // (N * 8 * 35)))  # a few GB of inputs in flight
    anc = synth.anchors_for(8)
    batch = Batch(L.MODEL_K8, N, device=local, anchors=anc, xml=synth.K8_XML, accel_noise=0.5, jolt=0.5)
    bufs = synth.k8_montecarlo_chunk(N, 0, chunk, anc, dev, seed=synth.SEED, full=full, first_filter=lo, want_x0=True,
                                     stream=stream)
    x0 = bufs["x0"].clone()
    batch.set_truth(bufs["truth_end"], stream=stream)  # rewritten in place by every chunk: the last one counts

    def step():
        nonlocal bufs
        batch.set_state(x0, None, stream=stream)
        for m0 in range(0, n_macro, chunk):
            bufs = synth.k8_montecarlo_chunk(N, m0, min(chunk, n_macro - m0), anc, dev, seed=synth.SEED, full=full,
                                             first_filter=lo, out=bufs, stream=stream)
            batch.replay_events(bufs["events"], ranges=bufs["ranges"], sensors=bufs["sensors"], err=0.01, stream=stream)
        batch.error_stats(stream=stream, readback=False)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
    for _ in range(W):
        step()
    batch.counters(reset=True)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(K):
        step()
    s = batch.stats_allreduce(comm, stream=stream)
    e1.record(stream)
    barrier()
    t = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    cnt = batch.counters(reset=True)
    if dump:
        dump_outputs(dump, batch, s, stream)
    batch.close()
    del bufs, x0
    torch.cuda.empty_cache()
    n_ev = n_macro * len(macro)
    return {"events_per_s": total_filters * n_ev * K / (ms * 1e-3), "toa_updates_per_s": total_filters * n_macro * K / (ms * 1e-3),
            "ms_per_step": ms / K, "steps": K, "warmup": W, "total_filters": total_filters, "filters_per_gpu": N,
            "n_gpus": world, "macro_steps": n_macro, "events_per_macro_step": len(macro), "chunk_macro_steps": chunk,
            "scaling": "strong", "rmse_xy_m": float(s[5]), "rmse_xy_hex": float(s[5]).hex(),
            "sum_e2_hex": float(s[0]).hex(), "filters_counted": float(s[2]), "bad_filters": float(s[3]),
            "bad_updates_this_rank": cnt["bad"],
            "data": "synthetic, generated on the device (Philox4x32-10) inside the timed region",
            "collective": "kfpos_stats_allreduce: one ncclAllGather of 4 doubles per rank + pairwise rank tree"}


def run_config5(args):
    """--workload config3 / config5: those BASELINE configs themselves as the whole job; prints its own JSON
    line (metric k8_multisensor_events_per_sec)."""
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ["NCCL_DEBUG"] = "WARN"
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    full = args.workload == "config5"
    if not args.mc_filters:
        args.mc_filters = (1 << 26) if full else (1 << 20)
    if not args.mc_macro_steps:
        args.mc_macro_steps = 4 if full else 1000
    comm = None
    if world > 1:
        from roskfpos_b200.shard import nccl_comm
        comm = nccl_comm(rank, world, local)
    r = config5_leg(local, dev, world, rank, comm, args.mc_filters, args.mc_macro_steps, args.steps, args.warmup, full=full,
                    dump=args.dump_outputs if rank == 0 else None)
    if rank == 0:
        print(json.dumps({"metric": "k8_multisensor_events_per_sec", "value": r["events_per_s"],
                          "unit": "events/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                          "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": "strong",
                          "vs_baseline": None, "dtype": "f64", "data": r["data"],
                          "config": {"workload": f"BASELINE config {'5: K8 (UWB+IMU+mag+PX4Flow)' if full else '3: K8 (UWB+IMU+compass)'} "
                                                 f"Monte Carlo, {args.mc_filters} filters in total, {args.mc_macro_steps} macro-steps of "
                                                 f"{r['events_per_macro_step']} events, 8 anchors",
                                     "filters_per_gpu": r["filters_per_gpu"], "chunk_macro_steps": r["chunk_macro_steps"],
                                     "parallelism": f"filters sharded by index over {world} GPU(s); {r['collective']}"},
                          "detail": r}))
    if comm is not None:
        comm.close()
    if world > 1:
        dist.destroy_process_group()


def bench_other_configs(local, dev, args):
    """The remaining BASELINE.json configs as secondary numbers (device-resident inputs, CUDA
    events, 1 warm-up + 3 timed repetitions each).  Not the headline metric."""
    import torch
    from roskfpos_b200 import lib as L, synth
    from roskfpos_b200.batch import Batch
    stream = torch.cuda.current_stream()
    out = {}

    def timed(fn, reps=3):
        fn()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        for _ in range(reps):
            fn()
        b.record(stream)
        torch.cuda.synchronize()
        return a.elapsed_time(b) / reps * 1e-3

    # ---- config 2: ML multilateration, 8 anchors, 1 Mi epochs (3-D from (1,1,4), and 2-D)
    N = 1 << 20
    anc = synth.anchors_for(8)
    r, _, _ = synth.device_ranges_mm(N, 1, anc, 0.1, dev, seed=synth.SEED + 5)
    r = r[0].contiguous()
    outs = dict(pos=torch.empty((3, N), device=dev, dtype=torch.float64),
                cov=torch.empty((9, N), device=dev, dtype=torch.float64),
                iters=torch.empty(N, device=dev, dtype=torch.int32),
                sel=torch.empty((2, N), device=dev, dtype=torch.int32),
                status=torch.empty(N, device=dev, dtype=torch.int32))
    for use2d in (0, 1):
        with Batch(L.MODEL_ML, N, device=local, anchors=anc, use2d=use2d,
                   ml_start=[1.0, 1.0, 1.0 if use2d else 4.0]) as b:
            t = timed(lambda: b.ml_solve(r, err=0.01, out=outs, stream=stream))
            c = b.counters()
        i_ml = c["ml_iters"] / max(c["updates"], 1)
        # SURVEY.md §8(d): ML standalone epoch = W_ml0 + I_ml W_mlit(d, m) + (15 + d + 1.5 d (d + 1)) m + (8 | 40)
        d, m = (2, 8) if use2d else (3, 8)
        w_epoch = ((12 * m if d == 2 else 0) + i_ml * ((46 * m + 25) if d == 2 else (59 * m + 60))
                   + (15 + d + 1.5 * d * (d + 1)) * m + (8 if d == 2 else 40))
        peak = C_double_peak(local)
        out[f"config2_ml_{'2d' if use2d else '3d'}"] = {
            "epochs_per_s": N / t, "ms": t * 1e3, "epochs": N, "anchors": 8, "mean_newton_iters": i_ml,
            "roofline": {"bound": "fp64", "achieved": w_epoch * N / t / 1e12, "peak": peak / 1e12, "unit": "TFLOP/s",
                         "frac": w_epoch * N / t / peak if peak else None, "flop_per_epoch": w_epoch,
                         "numerator": "SURVEY.md §8(d) W_alg of a standalone ML epoch with the measured Newton iterations",
                         "kernel": "ml_solve_kernel<false,8,false>" if use2d else "ml_stream3_kernel<8>",
                         "peak_source": "measured live: kfpos_measure_fp64_peak"}}
    # ---- config 4a/4b: NLOS variants, 16 anchors
    anc16 = synth.anchors_for(16)
    N4 = 1 << 22
    r16, _, _ = synth.device_ranges_mm(N4, 1, anc16, 0.1, dev, seed=synth.SEED + 6)
    r16 = r16[0].contiguous()
    o4 = dict(pos=torch.empty((3, N4), device=dev, dtype=torch.float64), cov=None, iters=None,
              sel=torch.empty((2, N4), device=dev, dtype=torch.int32), status=None)
    with Batch(L.MODEL_ML, N4, device=local, anchors=anc16, use2d=0, variant=1, num_ignored_rangings=2) as b:
        t = timed(lambda: b.ml_solve(r16, err=0.01, out=o4, stream=stream))
    out["config4a_ml_ignore2_16anchors"] = {"epochs_per_s": N4 / t, "ms": t * 1e3, "epochs": N4}
    # variant 2 (BestGroup, exact-order solver, a warp per epoch): the BASELINE size on the BASELINE geometry (the 4 x 4
    # grid, where the scan of most epochs ends at the first collinear triple the way the reference's exception
    # does), a jittered grid on which every epoch enumerates all 560 subsets, and the 3-D scan (1820 subsets of 4)
    import numpy as np
    jit = anc16.copy()
    jit[:, :2] += np.random.default_rng(3).uniform(-0.3, 0.3, size=(16, 2))
    rj, _, _ = synth.device_ranges_mm(1 << 20, 1, jit, 0.1, dev, seed=synth.SEED + 6)
    rj = rj[0].contiguous()
    for key, ranges, a, Nb, use2d in (("config4b_ml_best3_of_16_2d", r16, anc16, N4, 1),
                                      ("config4b_ml_best3_of_16_2d_jittered_grid", rj, jit, 1 << 20, 1),
                                      ("config4b_ml_best4_of_16_3d", r16, anc16, 1 << 17, 0)):
        ob = dict(pos=torch.empty((3, Nb), device=dev, dtype=torch.float64), cov=None, iters=None,
                  sel=torch.empty((2, Nb), device=dev, dtype=torch.int32), status=None)
        rb = ranges[:, :Nb].contiguous()
        with Batch(L.MODEL_ML, Nb, device=local, anchors=a, use2d=use2d, variant=2,
                   ml_start=[1.0, 1.0, 1.0 if use2d else 4.0]) as b:
            t = timed(lambda: b.ml_solve(rb, err=0.01, out=ob, stream=stream), reps=1)
            c = b.counters()
        out[key] = {"epochs_per_s": Nb / t, "ms": t * 1e3, "epochs": Nb,
                    "subsets_per_epoch": 560 if use2d else 1820,
                    "mean_newton_iters_per_epoch": c["ml_iters"] / max(c["updates"], 1),
                    "epochs_where_the_scan_throws": c["bad"] / max(c["updates"], 1)}
        del ob, rb
    del rj
    del r16, o4
    # ---- config 4c: T6 leave-one-out (ignoreWorstAnchorMode), 16 anchors
    Nl, Tl = 1 << 18, 10
    rl, x0l, _ = synth.device_ranges_mm(Nl, Tl, anc16, 0.1, dev, seed=synth.SEED + 7)
    x0f = torch.zeros((6, Nl), device=dev, dtype=torch.float64)
    x0f[:3] = x0l
    with Batch(L.MODEL_T6, Nl, device=local, anchors=anc16, accel_noise=0.5, ignore_worst_anchor=1,
               ignore_cost_threshold=0.5) as b:
        def run():
            b.set_state(x0f, None, stream=stream)
            b.replay_toa(0.1, rl, err=0.01, stream=stream)
        t = timed(run)
    out["config4c_t6_leave_one_out_16anchors"] = {"updates_per_s": Nl * Tl / t, "ms": t * 1e3,
                                                  "filters": Nl, "epochs": Tl, "solves_per_update": 17}
    # ---- config 4 (EKF side): variant 1, the 2 worst of 16 rangings dropped before the update
    with Batch(L.MODEL_T6, Nl, device=local, anchors=anc16, accel_noise=0.5, variant=1, num_ignored_rangings=2) as b:
        def run():
            b.set_state(x0f, None, stream=stream)
            b.replay_toa(0.1, rl, err=0.01, stream=stream)
        t = timed(run)
    out["config4_t6_variant1_ignore2_16anchors"] = {"updates_per_s": Nl * Tl / t, "ms": t * 1e3, "filters": Nl,
                                                    "epochs": Tl}
    del rl
    # ---- epoch assembler (SURVEY.md §8f-1): raw ranging logs -> epoch tensors; HBM-bound
    from roskfpos_b200.batch import assemble_epochs
    Na, n_seq, Ma = 1 << 19, 32, 8
    La = n_seq * Ma
    g = torch.Generator(device=dev); g.manual_seed(11)
    a_idx = torch.arange(La, device=dev, dtype=torch.int64).remainder(Ma).to(torch.uint8)[:, None].expand(La, Na).contiguous()
    sq = (torch.arange(La, device=dev) // Ma).to(torch.uint8)[:, None].expand(La, Na).contiguous()
    rmm = torch.randint(500, 15000, (La, Na), generator=g, device=dev, dtype=torch.int32)
    tt = (torch.arange(La, device=dev, dtype=torch.float64) * 0.002 + (torch.arange(La, device=dev) // Ma) * 0.084)[:, None] \
        .expand(La, Na).contiguous()
    Ta = n_seq + 2
    oa = dict(ranges=torch.empty((Ta, Ma, Na), dtype=torch.int32, device=dev), err=None,
              dt=torch.empty((Ta, Na), dtype=torch.float64, device=dev),
              n_epochs=torch.empty(Na, dtype=torch.int32, device=dev))
    t = timed(lambda: assemble_epochs(a_idx, sq, rmm, tt, Ma, Ta, fix_row_clear=True, device=local, out=oa, stream=stream))
    bytes_a = La * Na * (1 + 1 + 4 + 8) + Ta * Ma * Na * 4 + Ta * Na * 8 + Na * 4
    peaks, _ = load_peaks()
    out["assembler_fixed_row_clear"] = {"rangings_per_s": La * Na / t, "ms": t * 1e3, "logs": Na, "rangings_per_log": La,
                                        "algorithmic_gbs": bytes_a / t / 1e9,
                                        "hbm_frac": bytes_a / t / 1e9 / peaks["hbm_gbs"] if peaks.get("hbm_gbs") else None,
                                        "note": "includes the call's scratch allocation and stream sync"}
    del a_idx, sq, rmm, tt, oa
    # ---- configs 3 and 5: K8 multi-sensor event streams, 8 anchors, 1 Mi filters
    for name, full, n_macro in (("config3_k8_imu_mag", False, 5), ("config5_k8_full_multisensor", True, 4)):
        Nk = 1 << 20
        w = synth.k8_workload(Nk, n_macro, anc, seed=synth.SEED + 8, full=full, xp=torch, device=dev)
        with Batch(L.MODEL_K8, Nk, device=local, anchors=anc, xml=synth.K8_XML, accel_noise=0.5, jolt=0.5) as b:
            def run():
                b.set_state(w["x0"], None, stream=stream)
                b.replay_events(w["events"], ranges=w["ranges"], sensors=w["sensors"], err=0.01, stream=stream)
            t = timed(run)
            b.counters(reset=True)
            run()
            c = b.counters()
            s4 = b.error_stats(w["truth_end"], stream=stream)
        out[name] = {"toa_updates_per_s": Nk * w["n_toa"] / t, "all_event_updates_per_s": Nk * w["n_events"] / t,
                     "ms": t * 1e3, "filters": Nk, "events": w["n_events"], "toa_events": w["n_toa"],
                     "rmse_xy_m": float(np.sqrt(s4[1] / max(s4[2], 1))), "bad_updates": c["bad"],
                     "input_mb": (w["sensors"].numel() * 8 + w["ranges"].numel() * 4) / 1e6,
                     "roofline": k8_roofline(w["events"], full, 8, Nk, c, t, C_double_peak(local))}
        del w
    # ---- config 5 at scale: 8 Mi filters (the per-GPU share of the 64 M-filter Monte Carlo on 8 GPUs), inputs
    # synthesised on the device chunk by chunk (kfpos_synth_k8) and replayed; generation is inside the timed region
    torch.cuda.empty_cache()
    Nm, n_macro, chunk = 1 << 23, 8, 2
    with Batch(L.MODEL_K8, Nm, device=local, anchors=anc, xml=synth.K8_XML, accel_noise=0.5, jolt=0.5) as b:
        first = synth.k8_montecarlo_chunk(Nm, 0, chunk, anc, dev, seed=synth.SEED + 9, full=True, want_x0=True, stream=stream)
        x0m = first["x0"].clone()
        bufs = first

        def run_mc(replay=True):
            nonlocal bufs
            b.set_state(x0m, None, stream=stream)
            for m0 in range(0, n_macro, chunk):
                bufs = synth.k8_montecarlo_chunk(Nm, m0, chunk, anc, dev, seed=synth.SEED + 9, full=True, out=bufs, stream=stream)
                if replay:
                    b.replay_events(bufs["events"], ranges=bufs["ranges"], sensors=bufs["sensors"], err=0.01, stream=stream)
        t_all = timed(run_mc, reps=2)
        s4 = b.error_stats(bufs["truth_end"], stream=stream)
        c = b.counters()
        t_gen = timed(lambda: run_mc(False), reps=2)
    n_ev = n_macro * len(synth.MACRO_FULL)
    out["config5_k8_montecarlo_8Mi_filters"] = {
        "all_event_updates_per_s": Nm * n_ev / t_all, "toa_updates_per_s": Nm * n_macro / t_all, "ms": t_all * 1e3,
        "generation_ms": t_gen * 1e3, "filters": Nm, "events": n_ev, "chunk_macro_steps": chunk,
        "rmse_xy_m": float(np.sqrt(s4[1] / max(s4[2], 1))), "bad_updates": c["bad"],
        "note": "inputs generated in-kernel (Philox4x32-10) inside the timed region, never resident as a whole"}
    del bufs, first, x0m
    return out


def C_double_peak(device):
    import ctypes as C
    from roskfpos_b200 import lib as L
    v = C.c_double(0.0)
    L.check(L.lib().kfpos_measure_fp64_peak(int(device), C.byref(v)), "kfpos_measure_fp64_peak")
    return v.value


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--filters", type=int, default=1 << 20, help="filters per GPU")
    ap.add_argument("--tsteps", type=int, default=1000,
                    help="ranging epochs per bench step (1000: the 33.5 GB range log stays resident in HBM and a "
                         "20-step timed region lasts seconds, i.e. the number is a sustained one)")
    ap.add_argument("--e2e-tsteps", type=int, default=100, help="epochs of the pinned HOST log of the e2e leg")
    ap.add_argument("--anchors", type=int, default=8)
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the secondary BASELINE configs")
    ap.add_argument("--no-config5", action="store_true", help="skip the 64 Mi-filter strong-scaling leg")
    ap.add_argument("--config5-filters", type=int, default=1 << 26, help="TOTAL K8 filters of the config-5 leg")
    ap.add_argument("--workload", default="t6", choices=["t6", "config3", "config5"],
                    help="t6 = the headline metric (default); config3 / config5 = those BASELINE configs themselves: the "
                         "K8 IMU+compass+UWB (1 Mi filters x 1000 steps) / full multi-sensor (64 Mi filters) Monte Carlo "
                         "with --mc-filters filters in TOTAL sharded over the ranks (strong scaling)")
    ap.add_argument("--mc-filters", type=int, default=0, help="config3/5: total filters (default 1 Mi / 64 Mi)")
    ap.add_argument("--mc-macro-steps", type=int, default=0,
                    help="config3/5: 0.1 s macro-steps per bench step (default 1000 / 4)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="--impl b200: after the timed steps, write what the last one computed (state, covariance, "
                         "status of a fixed sample of rank 0's filters, reduced error statistics) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        # the reference leg times a sample whose size follows the measured CPU speed: nothing fixed to compare
        ap.error("--dump-outputs applies to --impl b200")
    if args.warmup < 3 and args.impl == "b200":
        args.warmup = max(args.warmup, 1)
    if args.impl == "reference":
        run_reference(args)
    elif args.workload in ("config3", "config5"):
        run_config5(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
