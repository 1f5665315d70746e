"""Where a small batch's forward time goes, and what narrow hGRU conv units change, through model.build only (so the
same script runs against a tree with or without narrow units).

    python monkey-pose_b200/csrc/devtools/small_batch.py --root TREE --tag NAME --out FILE --profile
    python monkey-pose_b200/csrc/devtools/small_batch.py --root TREE --tag NAME --out FILE [--dump DIR]
    python monkey-pose_b200/csrc/devtools/small_batch.py --merge FILE... --out FILE

--profile: one n = 1 forward per configuration under torch.profiler (CUDA activities), after a warm-up: per kernel
name its launches, summed device time and grid size (the stem, initial state, the 2T conv launches, fc_1, fc_out).
Run it in a process of its own; tracing slows the host.
Otherwise: frames/s and mean forward latency of model.build on device input at each n of NS, from one capacity-256
plan, CUDA events around >= 0.3 s of forwards, for k = 25 (T = 8), k = 64 (T = 8) and k = 32 (T = 16), bf16 and
fp16.  --dump DIR also saves the fp16 predictions at n = 256 (bench.py has no fp16 mode) for a bitwise comparison
of two builds.  Run old and new trees alternating in one session; --merge combines the per-run files with the
card's name and power limit (run it on the machine that measured)."""
import argparse
import json
import os
import subprocess
import sys

ap = argparse.ArgumentParser()
ap.add_argument("--root")
ap.add_argument("--tag")
ap.add_argument("--out", required=True)
ap.add_argument("--profile", action="store_true")
ap.add_argument("--dump")
ap.add_argument("--merge", nargs="*")
a = ap.parse_args()

if a.merge:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,driver_version",
                        "--format=csv,noheader"], capture_output=True, text=True).stdout.strip().splitlines()
    runs = [json.load(open(f)) for f in a.merge]
    json.dump({"gpu": q[0] if q else "unknown", "runs": runs}, open(a.out, "w"), indent=1)
    sys.exit(0)

sys.path.insert(0, os.path.abspath(a.root))
import numpy as np  # noqa: E402
import torch  # noqa: E402

import monkey_pose_b200 as mp  # noqa: E402
from monkey_pose_b200 import initialization as init  # noqa: E402

NS = (1, 2, 4, 8, 16, 32, 37, 64, 256)
CONFIGS = ((25, 8), (64, 8), (32, 16))
MODES = ("bf16", "fp16")
torch.cuda.set_device(0)
depth = torch.as_tensor(init.synthetic_depth(256, seed=1234)).cuda()
res = {"tag": a.tag, "root": os.path.basename(os.path.abspath(a.root)),
       "sms": torch.cuda.get_device_properties(0).multi_processor_count}


def model(k, T, mode):
    m = mp.model()
    m.channels, m.timesteps, m.compute_mode = k, T, mode
    m.load_params(init.pose_params(channels=k, S=15, T=T, hw=64, fc_hidden=1024, out=69, seed=3))
    m.build(depth, 69)      # capacity 256
    torch.cuda.synchronize()
    return m


def fps(m, n):
    d = depth[:n]
    for _ in range(3):
        m.build(d, 69)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    m.build(d, 69)
    e1.record()
    e1.synchronize()
    reps = max(5, int(0.3 / max(e0.elapsed_time(e1) / 1e3, 1e-5)))
    e0.record()
    for _ in range(reps):
        m.build(d, 69)
    e1.record()
    e1.synchronize()
    s = e0.elapsed_time(e1) / 1e3
    return {"fps": n * reps / s, "latency_ms": s / reps * 1e3}


if a.profile:
    from torch.profiler import ProfilerActivity, profile
    out = {}
    for k, T in CONFIGS:
        for mode in MODES:
            m = model(k, T, mode)
            d = depth[:1]
            for _ in range(5):
                m.build(d, 69)
            torch.cuda.synchronize()
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                m.build(d, 69)
                torch.cuda.synchronize()
            trace = os.path.join(os.path.dirname(os.path.abspath(a.out)), "trace_%s_k%d_%s.pt.trace.json" % (a.tag, k, mode))
            prof.export_chrome_trace(trace)
            kernels = {}
            ev = [e for e in json.load(open(trace))["traceEvents"] if e.get("cat") in ("kernel", "gpu_memcpy", "gpu_memset")]
            t0 = min(e["ts"] for e in ev)
            t1 = max(e["ts"] + e["dur"] for e in ev)
            for e in ev:
                r = kernels.setdefault(e["name"][:160], {"launches": 0, "us": 0.0, "grid": e.get("args", {}).get("grid")})
                r["launches"] += 1
                r["us"] += e["dur"]
            os.remove(trace)
            out["k%d_T%d_%s" % (k, T, mode)] = {"span_us": t1 - t0, "busy_us": sum(r["us"] for r in kernels.values()),
                                                "kernels": dict(sorted(kernels.items(), key=lambda kv: -kv[1]["us"]))}
            del m
    res["profile_n1"] = out
else:
    out = {}
    for k, T in CONFIGS:
        for mode in MODES:
            m = model(k, T, mode)
            out["k%d_T%d_%s" % (k, T, mode)] = {str(n): fps(m, n) for n in NS}
            if a.dump and mode == "fp16":
                os.makedirs(a.dump, exist_ok=True)
                pred = m.build(depth, 69)
                np.save(os.path.join(a.dump, "fp16_k%d_T%d_%s.npy" % (k, T, a.tag)), pred.float().cpu().numpy())
            del m
            torch.cuda.synchronize()
    res["throughput"] = out

json.dump(res, open(a.out, "w"), indent=1)
print(json.dumps(res)[:2000])
