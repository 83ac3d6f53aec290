#!/usr/bin/env python
"""A / B of builds of the library on the T6 headline step (bench.py, 1 Mi filters x 1000 epochs x 8 anchors, int32
resident): every build runs `bench.py --no-cpu --no-e2e --no-extra --no-config5 --dump-outputs` once per round, the
builds alternate, and the dumped outputs (x, P, status, error statistics) and the bench line's rmse_m, bad_updates and
roofline.mean_iters are compared byte for byte with the first build's.

    python profiles/t6_icache_ab.py OUT.json DUMPDIR ROUNDS NAME=LIB.so [NAME=LIB.so ...]
"""
import glob
import json
import os
import subprocess
import sys

out, dumpdir, rounds, builds = sys.argv[1], sys.argv[2], int(sys.argv[3]), [a.split("=", 1) for a in sys.argv[4:]]
root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                      capture_output=True, text=True).stdout.strip().splitlines()
res = {"card": card[0] if card else None, "command": "bench.py --gpus 1 --steps 10 --warmup 3 --no-cpu --no-e2e --no-extra "
       "--no-config5 --dump-outputs DIR", "runs": {n: [] for n, _ in builds}}
for r in range(rounds):
    for name, so in builds:
        d = os.path.join(dumpdir, f"{name}_{r}")
        env = dict(os.environ, KFPOS_B200_SO=os.path.abspath(so))
        p = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--gpus", "1", "--steps", "10", "--warmup", "3",
                            "--no-cpu", "--no-e2e", "--no-extra", "--no-config5", "--dump-outputs", d],
                           capture_output=True, text=True, env=env, cwd=root)
        lines = [ln for ln in p.stdout.splitlines() if ln.startswith("{")]
        if p.returncode or not lines:
            sys.exit(f"{name}: exit {p.returncode}\n{p.stdout[-2000:]}\n{p.stderr[-4000:]}")
        b = json.loads(lines[-1])
        run = {"value": b["value"], "ms_per_step": b["ms_per_step"], "rmse_m": b.get("rmse_m"),
               "bad_updates": b.get("bad_updates"), "mean_iters": b.get("roofline", {}).get("mean_iters")}
        res["runs"][name].append(run)
        print(name, r, json.dumps(run), flush=True)
ref = builds[0][0]
res["summary"] = {}
for name, _ in builds:
    v = [x["value"] for x in res["runs"][name]]
    ms = [x["ms_per_step"] for x in res["runs"][name]]
    same_line = all(x[k] == res["runs"][ref][0][k] for x in res["runs"][name] for k in ("rmse_m", "bad_updates", "mean_iters"))
    same_files = True
    for f in sorted(glob.glob(os.path.join(dumpdir, f"{ref}_0", "*.npy"))):
        for r in range(rounds):
            g = os.path.join(dumpdir, f"{name}_{r}", os.path.basename(f))
            same_files &= os.path.exists(g) and open(f, "rb").read() == open(g, "rb").read()
    res["summary"][name] = {"mean_value": sum(v) / len(v), "mean_ms_per_step": sum(ms) / len(ms),
                            "spread_pct": 100.0 * (max(ms) - min(ms)) / min(ms),
                            "speedup_vs_" + ref: (sum(v) / len(v)) / (sum(x["value"] for x in res["runs"][ref]) / rounds),
                            "outputs_identical_to_" + ref: bool(same_files), "bench_fields_identical_to_" + ref: same_line}
with open(out, "w") as fh:
    json.dump(res, fh, indent=1)
print(json.dumps(res["summary"], indent=1))
