"""Measure what running a batch below a plan's capacity saves, through model.build only (so the same script runs
against a tree with or without capacity-keyed plans).

    python monkey-pose_b200/csrc/devtools/batch_capacity.py --root TREE --tag NAME --out FILE [--throughput]
    python monkey-pose_b200/csrc/devtools/batch_capacity.py --merge FILE... --out FILE

rebuild: wall time of model.build + synchronize over the batch sequence 256, 200, 256, 1, 256 (k = 25 and k = 64,
bf16, the seeded random initial state), the first build (plan creation at 256) excluded.  A tree that keys its plan
on the batch re-creates the plan, re-packs the weights and re-draws the initial state at every change.
throughput (--throughput): frames/s of model.build on device input at n in {1, 8, 64, 200, 256}, from one
capacity-256 plan and from a dedicated plan per n, alternating, two rounds; CUDA events around >= 0.5 s of forwards.
--merge combines the per-run files with the card's name and power limit; run it on the machine that measured,
right after the runs."""
import argparse
import json
import os
import subprocess
import sys
import time

ap = argparse.ArgumentParser()
ap.add_argument("--root")
ap.add_argument("--tag")
ap.add_argument("--out", required=True)
ap.add_argument("--throughput", action="store_true")
ap.add_argument("--merge", nargs="*")
a = ap.parse_args()

if a.merge:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,driver_version",
                        "--format=csv,noheader"], capture_output=True, text=True).stdout.strip().splitlines()
    runs = [json.load(open(f)) for f in a.merge]
    json.dump({"gpu": q[0] if q else "unknown", "runs": runs}, open(a.out, "w"), indent=1)
    sys.exit(0)

sys.path.insert(0, os.path.abspath(a.root))
import torch  # noqa: E402

import monkey_pose_b200 as mp  # noqa: E402
from monkey_pose_b200 import initialization as init  # noqa: E402

SEQ = (256, 200, 256, 1, 256)
NS = (1, 8, 64, 200, 256)
torch.cuda.set_device(0)
depth = torch.as_tensor(init.synthetic_depth(256, seed=1234)).cuda()
res = {"tag": a.tag, "root": os.path.basename(os.path.abspath(a.root)), "rebuild": {}, "throughput": {}}


def model(k):
    m = mp.model()
    m.channels, m.timesteps, m.compute_mode = k, 8, "bf16"
    m.load_params(init.pose_params(channels=k, S=15, T=8, hw=64, fc_hidden=1024, out=69, seed=3))
    return m


for k in (25, 64):
    m = model(k)
    steps = []
    for i, n in enumerate(SEQ):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        m.build(depth[:n], 69)
        torch.cuda.synchronize()
        steps.append(time.perf_counter() - t0)
    res["rebuild"]["k%d" % k] = {"sequence": SEQ, "build_s": steps, "total_s_excl_first": sum(steps[1:])}
    del m
    torch.cuda.synchronize()


def fps(m, n):
    d = depth[:n]
    for _ in range(3):
        m.build(d, 69)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    m.build(d, 69)
    torch.cuda.synchronize()
    reps = max(5, int(0.5 / max(time.perf_counter() - t0, 1e-5)))
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        m.build(d, 69)
    e1.record()
    e1.synchronize()
    return n * reps / (e0.elapsed_time(e1) / 1e3)


if a.throughput:
    for k in (25, 64):
        cap = model(k)
        cap.build(depth, 69)
        out = {}
        for n in NS:
            out[str(n)] = {"capacity_256": [], "dedicated": []}
            for _ in range(2):
                out[str(n)]["capacity_256"].append(fps(cap, n))
                ded = model(k)
                out[str(n)]["dedicated"].append(fps(ded, n))
                del ded
        res["throughput"]["k%d" % k] = out
        del cap
        torch.cuda.synchronize()

json.dump(res, open(a.out, "w"), indent=1)
print(json.dumps(res))
