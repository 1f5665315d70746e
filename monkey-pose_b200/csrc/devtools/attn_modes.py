"""The attention CNN's two compute modes side by side: 'bf16x3' (bf16 hi/lo operand splits, three MMAs per k-step) and
'fp16' (one fp16 MMA per k-step), at the reference widths (64 .. 1024, fc 1024) on 424 x 512 frames.

    python monkey-pose_b200/csrc/devtools/attn_modes.py --out FILE [--rounds 3] [--window 1.0]
    python monkey-pose_b200/csrc/devtools/attn_modes.py --profile --out FILE

Timing: the modes alternate for --rounds rounds; each number is one window of >= --window seconds between CUDA events,
after a warm-up of the same call:
  attention ms per 256 frames: attn_model_struct.build at n = 256, and 256 single-frame builds (n = 1) on the same
    capacity-256 plan;
  FramesToJoints frames/s at batch 256 with the attention output driving the crop (no fixed centres), fed
    device-resident float32 frames and raw 16-bit frames from pinned host memory (upload in 4 pieces).
Agreement of fp16 with bf16x3 on the same 256 frames: the share of frames whose crop-window integers differ, the
invalid-window counts, the attention outputs' difference in pixels / mm, and the joints' difference in mm.  The pose
network is bench.py's (k = 25, T = 8, bf16).
Frames: 256 distinct scenes, an ellipsoidal object at a random place (rows / columns 0.2 .. 0.8 of the frame) and depth
(1.2 .. 2.8 m) in front of a noisy back wall 3.2 .. 4 m away, 5 % dropout pixels.  Head: random-init weights at the
reference widths, with afc_out calibrated per output (one scale, one bias) so that the bf16x3 centres over these frames
have mean (0.5, 0.5, 0.2) and standard deviation (0.12, 0.12, 0.03) of (height, width, 10 m): centres that move over
the frame by about 50 px and 300 mm, as a trained head's do.  Scaling the head scales the fp16 error at its output
with the spread, so the centre and window differences are those of a head with that spread.  The GEMM layers are
untouched.  The card's name and power limit are read in the same process.
--profile: torch.profiler (CUDA activities) over one attention build per mode at n = 256 and at n = 1, after a
warm-up: per kernel its launches and summed device time.  Run it in a process of its own; tracing slows the host."""
import argparse
import json
import os
import subprocess
import sys

ap = argparse.ArgumentParser()
ap.add_argument("--out", required=True)
ap.add_argument("--rounds", type=int, default=3)
ap.add_argument("--window", type=float, default=1.0, help="seconds per timed window")
ap.add_argument("--profile", action="store_true")
a = ap.parse_args()

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "..", ".."))
import numpy as np  # noqa: E402
import torch  # noqa: E402

import monkey_pose_b200 as mp  # noqa: E402
from monkey_pose_b200 import initialization as init  # noqa: E402
from monkey_pose_b200 import tf_monkeydetector as tmd  # noqa: E402

MODES = ("bf16x3", "fp16")
B, H, W = 256, 424, 512
torch.cuda.set_device(0)
q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,driver_version", "--format=csv,noheader",
                    "-i", "0"], capture_output=True, text=True).stdout.strip()
res = {"gpu": q or "unknown", "sms": torch.cuda.get_device_properties(0).multi_processor_count, "batch": B,
       "frame": [H, W]}


class Cfg(object):
    image_orig_size = [H, W, 1]
    image_target_size = [128, 128, 1]
    image_max_depth = 10000.


def scenes(n, seed):
    """n distinct depth frames / 10 m: an ellipsoidal object in front of a noisy back wall, 5 % dropout pixels"""
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:H, 0:W].astype(np.float32)
    out = np.empty((n, H, W), np.float32)
    for i in range(n):
        f = rng.uniform(3200, 4000) + rng.normal(0, 20, (H, W))
        cy, cx, d = rng.uniform(0.2, 0.8) * H, rng.uniform(0.2, 0.8) * W, rng.uniform(1200, 2800)
        ry, rx = rng.uniform(40, 90), rng.uniform(30, 70)
        r2 = ((yy - cy) / ry) ** 2 + ((xx - cx) / rx) ** 2
        f = np.where(r2 < 1, d - 150 * np.sqrt(np.clip(1 - r2, 0, 1)), f)
        f[rng.uniform(size=(H, W)) < 0.05] = 0
        out[i] = np.round(f) / 10000.0
    return out


CENTRE_MEAN, CENTRE_STD = np.array([0.5, 0.5, 0.2]), np.array([0.12, 0.12, 0.03])
frames_np = scenes(B, 99)
frames_dev = torch.as_tensor(frames_np).cuda()
raw_pin = torch.from_numpy(np.round(frames_np * 10000.0).astype(np.uint16).view(np.int16)).pin_memory()

# afc_out calibrated on the bf16x3 forward: tr = s * raw + b per output
P = dict(init.attn_params(seed=8))
P["afc_out/afc_out_biases"] = np.zeros(3, np.float32)
cal = mp.attn_model_struct()
cal.load_params(P)
raw = cal.build(frames_dev, 3).double().cpu().numpy()
del cal
scale = CENTRE_STD / raw.std(axis=0)
P["afc_out/afc_out_weights"] = (P["afc_out/afc_out_weights"] * scale).astype(np.float32)
P["afc_out/afc_out_biases"] = (CENTRE_MEAN - scale * raw.mean(axis=0)).astype(np.float32)
res["head"] = {"centre_mean": CENTRE_MEAN.tolist(), "centre_std": CENTRE_STD.tolist(), "afc_out_scale": scale.tolist()}
attn, md, pipe = {}, {}, {}
pm = mp.model()
pm.channels, pm.timesteps, pm.compute_mode = 25, 8, "bf16"
pm.hidden_state = torch.as_tensor(init.hidden_init((B, 64, 64, 25), seed=5)).cuda()
pm.load_params(init.pose_params(channels=25, S=15, T=8, hw=64, fc_hidden=1024, out=69, seed=3))
for mode in MODES:
    attn[mode] = mp.attn_model_struct()
    attn[mode].compute_mode = mode
    attn[mode].load_params(P)
    attn[mode].build(frames_dev, 3)                   # capacity 256
    md[mode] = tmd.tfMonkeyDetector(365.456, 365.456, 256, 212, [800, 800, 1200], 200, 10000)
    pipe[mode] = mp.FramesToJoints(attn[mode], pm, md[mode], Cfg(), cube_z=1200.0, chunks=4)
torch.cuda.synchronize()


def window(fn):
    """ms per call over >= a.window seconds between CUDA events, after a warm-up call"""
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    e1.synchronize()
    reps = max(3, int(a.window / max(e0.elapsed_time(e1) * 1e-3, 1e-6)) + 1)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / reps


if a.profile:
    from torch.profiler import ProfilerActivity, profile
    out = {}
    for mode in MODES:
        for n in (B, 1):
            d = frames_dev[:n]
            for _ in range(3):
                attn[mode].build(d, 3)
            torch.cuda.synchronize()
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                attn[mode].build(d, 3)
                torch.cuda.synchronize()
            trace = os.path.join(os.path.dirname(os.path.abspath(a.out)), "trace_attn_%s_n%d.pt.trace.json" % (mode, n))
            prof.export_chrome_trace(trace)
            kernels = {}
            for e in json.load(open(trace))["traceEvents"]:
                if e.get("cat") in ("kernel", "gpu_memcpy", "gpu_memset"):
                    r = kernels.setdefault(e["name"][:160], {"launches": 0, "us": 0.0})
                    r["launches"] += 1
                    r["us"] += e["dur"]
            os.remove(trace)
            out["%s_n%d" % (mode, n)] = {
                "busy_us": sum(r["us"] for r in kernels.values()),
                "kernels": dict(sorted(kernels.items(), key=lambda kv: -kv[1]["us"]))}
    res["profile"] = out
else:
    rounds = []
    for r in range(a.rounds):
        row = {}
        for mode in (MODES if r % 2 == 0 else MODES[::-1]):
            am, pp = attn[mode], pipe[mode]
            d1 = frames_dev[:1]

            def single():
                for _ in range(B):
                    am.build(d1, 3)

            row[mode] = {
                "attn_ms_per_256_n256": window(lambda: am.build(frames_dev, 3)),
                "attn_ms_per_256_n1": window(single),
                "f2j_fps_device_float": B / (window(lambda: pp(frames_dev)) * 1e-3),
                "f2j_fps_host_raw16": B / (window(lambda: pp(raw_pin)) * 1e-3),
            }
        rounds.append(row)
        print(json.dumps(row))
    res["rounds"] = rounds
    res["median"] = {m: {k: float(np.median([r[m][k] for r in rounds])) for k in rounds[0][m]} for m in MODES}
    # agreement on the same frames, attention output driving the crop
    got = {}
    for mode in MODES:
        tr = attn[mode].build(frames_dev, 3).double().cpu().numpy()
        xyz, _ = pipe[mode](frames_dev)
        got[mode] = (tr, xyz.double().numpy(), md[mode]._last_windows_dev[0].cpu().numpy(),
                     md[mode].last_invalid_dev.cpu().numpy())
    tr3, xyz3, win3, inv3 = got["bf16x3"]
    tr16, xyz16, win16, inv16 = got["fp16"]
    dtr = np.abs(tr16 - tr3) * np.array([H, W, 10000.0])
    jd = np.linalg.norm(xyz16 - xyz3, axis=2)
    same = (win16 == win3).all(axis=1)
    res["agreement"] = {
        "frames": B,
        "bf16x3_centre_spread": {"u_px_std": float(tr3[:, 0].std() * H), "v_px_std": float(tr3[:, 1].std() * W),
                                 "d_mm_std": float(tr3[:, 2].std() * 10000.0),
                                 "u_px_range": [float(tr3[:, 0].min() * H), float(tr3[:, 0].max() * H)],
                                 "v_px_range": [float(tr3[:, 1].min() * W), float(tr3[:, 1].max() * W)],
                                 "d_mm_range": [float(tr3[:, 2].min() * 1e4), float(tr3[:, 2].max() * 1e4)]},
        "window_ints_differ_share": float(1.0 - same.mean()),
        "invalid_windows": {"bf16x3": int((inv3 != 0).sum()), "fp16": int((inv16 != 0).sum())},
        "fp16_invalid_where_bf16x3_valid": int(((inv3 == 0) & (inv16 != 0)).sum()),
        "centre_diff": {"u_px_mean": float(dtr[:, 0].mean()), "u_px_max": float(dtr[:, 0].max()),
                        "v_px_mean": float(dtr[:, 1].mean()), "v_px_max": float(dtr[:, 1].max()),
                        "d_mm_mean": float(dtr[:, 2].mean()), "d_mm_max": float(dtr[:, 2].max())},
        "joint_diff_mm": {"mean": float(jd.mean()), "max": float(jd.max()),
                          "mean_same_window": float(jd[same].mean()) if same.any() else None,
                          "max_same_window": float(jd[same].max()) if same.any() else None},
    }

json.dump(res, open(a.out, "w"), indent=1)
print(json.dumps({k: v for k, v in res.items() if k != "profile"})[:3000])
