"""Speed and accuracy of the tensor-core compute modes side by side: bf16, fp16 and bf16x3 pose forwards at batch 256
for (k, T) = (25, 8), (64, 8) and (32, 16), in one process on one GPU.

Per workload the three modes get identical seeded inputs and parameters.  Timing: after a warm-up, the modes take
turns (--repeats rounds), each round timing >= --window-s seconds of back-to-back device-resident forwards with CUDA
events, so a drift of clock or load hits every mode alike.  After each window one more forward runs with kernel
timing on, to read the SM clock the conv kernels ran at (pose_plan_sm_clock_ghz: clock64 / %globaltimer inside the
kernel; the nominal clock nvidia-smi reports is not it under a power limit).  Accuracy: out_put and the hGRU output of
the same batch against the fp64 oracle on --oracle-frames frames (rel = max|a-b| / max|b|; mean joint deviation, mm).
Prints one JSON line.
    python monkey-pose_b200/csrc/devtools/mode_table.py [--out profiles/<name>.json]"""
import argparse
import ctypes
import json
import math
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "..", ".."))
import torch  # noqa: E402

import monkey_pose_b200 as mp  # noqa: E402
from monkey_pose_b200 import initialization as init  # noqa: E402
from oracle import hgru_oracle_np as onp  # noqa: E402
from oracle import hgru_oracle_torch as otorch  # noqa: E402

MODES = ("bf16", "fp16", "bf16x3")
WORKLOADS = ((25, 8), (64, 8), (32, 16))


def gpu_info():
    info = {"gpu": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm",
                            "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=30).stdout
        pl, clk = [x.strip() for x in q.strip().splitlines()[0].split(",")]
        info["power_limit_w"], info["sm_clock_max_mhz"] = float(pl), float(clk)
    except Exception as e:      # (reported, not guessed)
        info["power_limit_w"] = "unavailable: %s" % e
    return info


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--window-s", type=float, default=1.0)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--oracle-frames", type=int, default=2)
    ap.add_argument("--out", default=None, help="also write the JSON result to this file")
    a = ap.parse_args()
    assert torch.cuda.is_available(), "mode_table.py measures on a CUDA device"
    torch.cuda.set_device(0)
    lib = mp._lib.load()
    B = a.batch
    result = dict(gpu_info(), batch=B, repeats=a.repeats, window_s=a.window_s, workloads=[])
    for k, T in WORKLOADS:
        P = init.pose_params(channels=k, S=15, T=T, hw=64, fc_hidden=1024, out=69, seed=3)
        depth_np = init.synthetic_depth(B, seed=1234, size=128)
        h0_np = init.hidden_init((B, 64, 64, k), seed=5)
        depth = torch.as_tensor(depth_np).cuda()
        idx = list(range(a.oracle_frames))
        ref, acts = otorch.pose_forward(depth_np[idx], P, h0_np[idx], timesteps=T, dtype=torch.float64, trace=True)
        ref, ref_h = ref.numpy(), acts["hgru"].numpy()
        models, row = {}, {"k": k, "T": T, "modes": {}}
        for mode in MODES:
            m = mp.model()
            m.channels, m.timesteps, m.compute_mode = k, T, mode
            m.hidden_state = torch.as_tensor(h0_np).cuda()
            m.load_params(P)
            out = m.build(depth, 69).cpu().numpy()
            got_h = m.activation("hgru").cpu().numpy()[idx]
            for _ in range(a.warmup):
                m.build(depth, 69)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(3):
                m.build(depth, 69)
            e1.record()
            torch.cuda.synchronize()
            steps = max(3, math.ceil(a.window_s * 1000.0 / (e0.elapsed_time(e1) / 3)))
            models[mode] = (m, steps)
            row["modes"][mode] = {
                "out_rel_err": onp.rel_err(out[idx], ref)[0], "hgru_rel_err": onp.rel_err(got_h, ref_h)[0],
                "mean_joint_dev_mm": onp.mean_joint_error_mm(out[idx], ref), "steps_per_window": steps,
                "fps": [], "window_s": [], "sm_clock_in_kernel_ghz": []}
        for _ in range(a.repeats):
            for mode in MODES:
                m, steps = models[mode]
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(steps):
                    m.build(depth, 69)
                e1.record()
                torch.cuda.synchronize()
                ms = e0.elapsed_time(e1)
                lib.hgru_enable_kernel_timing(1)
                m.build(depth, 69)
                g_mean, g_min = ctypes.c_float(0), ctypes.c_float(0)
                lib.pose_plan_sm_clock_ghz(m._plan, ctypes.byref(g_mean), ctypes.byref(g_min))
                lib.hgru_enable_kernel_timing(0)
                r = row["modes"][mode]
                r["fps"].append(round(B * steps / (ms / 1000.0), 1))
                r["window_s"].append(round(ms / 1000.0, 3))
                r["sm_clock_in_kernel_ghz"].append(round(float(g_mean.value), 4))
        for mode in MODES:
            r = row["modes"][mode]
            r["fps_median"] = statistics.median(r["fps"])
            r["fps_spread_pct"] = round(100.0 * (max(r["fps"]) - min(r["fps"])) / r["fps_median"], 2)
        bf, fp = row["modes"]["bf16"], row["modes"]["fp16"]
        # paired by round: the two modes ran back to back
        row["fp16_over_bf16_fps"] = [round(x / y, 4) for x, y in zip(fp["fps"], bf["fps"])]
        row["fp16_over_bf16_fps_median"] = statistics.median(row["fp16_over_bf16_fps"])
        row["fp16_over_bf16_hgru_err"] = round(fp["hgru_rel_err"] / bf["hgru_rel_err"], 4)
        row["fp16_over_bf16_out_err"] = round(fp["out_rel_err"] / bf["out_rel_err"], 4)
        result["workloads"].append(row)
        print("k=%d T=%d: " % (k, T) + ", ".join(
            "%s %.0f fps (spread %.1f %%) out rel %.2e hgru rel %.2e %.4f mm" % (
                md, row["modes"][md]["fps_median"], row["modes"][md]["fps_spread_pct"], row["modes"][md]["out_rel_err"],
                row["modes"][md]["hgru_rel_err"], row["modes"][md]["mean_joint_dev_mm"]) for md in MODES),
            file=sys.stderr)
        del models
        torch.cuda.empty_cache()
    line = json.dumps(result)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
