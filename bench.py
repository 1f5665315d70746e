#!/usr/bin/env python
"""bench.py -- depth frames/sec of the hGRU-pose forward (8 timesteps, 15x15 horizontal kernels).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

One "step" = one forward pass of the whole hot path (stem -> 8-step hGRU -> readout) over one batch
of synthetic 128x128 depth crops.  Workload at every N: BASELINE.json configs[1] per GPU (batch 256,
25 hidden channels, 15x15, T = 8), i.e. weak scaling; frames are sharded over ranks with no
data-path collective, predictions are all-gathered (NCCL) at the end of each step.

Prints ONE JSON line on rank 0 (see the contract in the task statement): `value` is device-resident
throughput, `e2e` the same metric through the public API with pinned host buffers (H2D + D2H inside
the timed region), `roofline` the tensor-pipe fraction of the dominant kernel (the tcgen05
horizontal conv) timed live with CUDA events, `cpu_baseline` the torch-CPU oracle on a bounded sample.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "depth frames/sec (hGRU 8-step fwd)"
UNIT = "frames/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=256, help="frames per GPU per step")
    ap.add_argument("--channels", type=int, default=25)
    ap.add_argument("--timesteps", type=int, default=8)
    ap.add_argument("--mode", default="bf16", choices=["bf16", "fp32", "bf16x3"],
                    help="bf16: tcgen05, bf16 operands; bf16x3: tcgen05, bf16 hi/lo splits (fp32-class, k <= 32); "
                         "fp32: exact SIMT")
    ap.add_argument("--cpu-frames", type=int, default=64, help="frames in the CPU-baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-stages", action="store_true", help="skip the crop / post-processing stage timings")
    ap.add_argument("--no-extra", action="store_true", help="skip the short runs of the other BASELINE configs")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the predictions of the last timed step to DIR/out_put.npy (float32), so that two "
                         "builds can be compared output for output on the same seeded inputs")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    return a


DUMP_LIMIT_BYTES = 64 << 20


def dump_output(directory, name, x):
    """Writes x as DIR/<name>.npy in float32.  An output larger than DUMP_LIMIT_BYTES (many ranks' gathered
    predictions) is cut to a fixed, seeded sample of its rows, whose sorted indices go to DIR/<name>_rows.npy."""
    import numpy as np
    os.makedirs(directory, exist_ok=True)
    x = np.ascontiguousarray(x, dtype=np.float32)
    if x.nbytes > DUMP_LIMIT_BYTES:
        n_rows = DUMP_LIMIT_BYTES // (x[:1].nbytes + 8)          # + 8 bytes per row for its float64 index
        rows = np.sort(np.random.default_rng(0).choice(len(x), n_rows, replace=False))
        x = x[rows]
        np.save(os.path.join(directory, name + "_rows.npy"), rows.astype(np.float64))
    np.save(os.path.join(directory, name + ".npy"), x)


def config_label(batch, channels, timesteps):
    """Which BASELINE.json config (if any) a (per-GPU batch, channels, timesteps) triple is."""
    if (channels, timesteps) == (25, 8):
        return "BASELINE configs[1]" if batch == 256 else \
            ("BASELINE configs[2] per-GPU shard" if batch == 512 else "BASELINE configs[4] sweep point")
    if (channels, timesteps) == (32, 16):
        return "BASELINE configs[3], the deep variant"
    if (channels, timesteps) == (64, 8):
        return "the reference's own width, hgru_pose.py:50-81"
    return "non-BASELINE sweep point"


def workload_config(a, n_gpus):
    return {"workload": "hgru_pose forward, batch %d per GPU, 128x128 crops, 15x15 h-kernels, %d hidden "
                        "channels, T=%d (%s)" % (a.batch, a.channels, a.timesteps,
                                                 config_label(a.batch, a.channels, a.timesteps)),
            "global_batch": a.batch * n_gpus, "per_gpu_batch": a.batch, "channels": a.channels,
            "timesteps": a.timesteps, "h_kernel": 15, "hconv_arithmetic": a.mode,
            "parallelism": "batch-sharded x%d, no data-path collective" % n_gpus + (
                "; predictions all-gathered every step, asynchronously (complete inside the timed region)"
                if n_gpus > 1 else ""),
            "cache": "per-step working set (%.0f MB of fp32 state per tensor) exceeds the 126 MB L2"
                     % (a.batch * 64 * 64 * max(16, (a.channels + 15) // 16 * 16) * 4 / 1e6)}


# ------------------------------------------------------------------------------------------------
# CPU arm: the oracle port (torch-CPU stand-in for the reference's TF-CPU forward; TF is absent)
# ------------------------------------------------------------------------------------------------
def cpu_forward_fps(a, frames, reps):
    import torch
    from monkey_pose_b200 import initialization as init
    from oracle import hgru_oracle_torch as otorch
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    P = init.pose_params(channels=a.channels, S=15, T=a.timesteps, hw=64, fc_hidden=1024, out=69, seed=3)
    P = {k: torch.as_tensor(v) for k, v in P.items()}
    depth = init.synthetic_depth(frames, seed=1234)
    h0 = init.hidden_init((frames, 64, 64, a.channels), seed=5)
    otorch.pose_forward(depth[:2], P, h0[:2], timesteps=a.timesteps)      # warm-up
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        otorch.pose_forward(depth, P, h0, timesteps=a.timesteps)
        ts.append(time.perf_counter() - t0)
    ts.sort()
    med = ts[len(ts) // 2]
    return frames / med, med, cores


def run_reference(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps = max(1, a.steps)
    # (cpu_forward_fps runs one untimed 2-frame forward first: thread pool and oneDNN primitives are warm; a full
    # --warmup W of 64-frame CPU forwards would not fit the few-minutes budget of this arm)
    fps, med, cores = cpu_forward_fps(a, a.cpu_frames, steps)
    sample = "%d frames per step (of the %d-frame batch), median of %d steps" % (a.cpu_frames, a.batch, steps)
    line = {"impl": "reference", "metric": METRIC, "value": fps, "unit": UNIT, "n_gpus": a.gpus,
            "steps": steps, "warmup": a.warmup, "ms_per_step": med * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(a, a.gpus),
            "cpu_baseline": {"value": fps, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample,
                             "note": "torch-CPU oracle: TensorFlow 1.x / Python 2 reference cannot run"},
            "e2e": {"value": fps, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------
# clocks sampler (nvidia-smi during the timed region)
# ------------------------------------------------------------------------------------------------
class Clocks(object):
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                 "-lms", "10"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def wait_ready(self, timeout=4.0):
        """nvidia-smi needs ~0.1-1 s before its first row: do not enter a 50 ms timed region before it samples."""
        t = time.perf_counter()
        while self.proc is not None and not self.rows and time.perf_counter() - t < timeout:
            time.sleep(0.01)

    def _read(self):
        for ln in self.proc.stdout:
            self.rows.append((time.perf_counter(), ln.strip()))

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons, pw, allrows = [], None, set(), [], []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ts, ln in self.rows:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                c, m = float(f[0]), float(f[1])
            except ValueError:
                continue
            mx = m
            allrows.append((ts, c))
            if t0 <= ts <= t1 + 0.02:
                sm.append(c)
                try:
                    pw.append(float(f[2]))
                except ValueError:
                    pass
                for nme, v in zip(names, f[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(nme)
        if not sm and allrows:      # timed region shorter than the sampling period: nearest sample
            mid = 0.5 * (t0 + t1)
            sm = [min(allrows, key=lambda r: abs(r[0] - mid))[1]]
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm), "power_w_max": max(pw) if pw else None}


# ------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------
def run_ours(a):
    import ctypes
    import torch
    import torch.distributed as dist
    import monkey_pose_b200 as mp
    from monkey_pose_b200 import initialization as init
    from monkey_pose_b200.sharding import PredictionGatherer

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs CUDA devices (there is no CPU fallback)"
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    n_gpus = world
    lib = mp._lib.load()
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = peaks.get("bf16_tflops_sustained") or 1400.0
    peak_burst = peaks.get("bf16_tflops") or 1650.0
    peak_src = "MEASURED_PEAKS.json bf16_tflops_sustained (kernel timed inside a long step)" \
        if "bf16_tflops_sustained" in peaks else "fallback 1.4 PFLOP/s sustained (B200_PROFILING.md)"

    def sync():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def timed(fn, steps, drain=None):
        sync()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record()
        for _ in range(steps):
            fn()
        if drain is not None:
            drain()              # collectives still in flight are part of the job: the stream waits for them here
        e1.record()
        sync()
        t1 = time.perf_counter()
        ms = e0.elapsed_time(e1)
        t = torch.tensor([ms], device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()), t0, t1

    def make_model(channels, timesteps, mode, B, seed_off):
        P = init.pose_params(channels=channels, S=15, T=timesteps, hw=64, fc_hidden=1024, out=69, seed=3)
        h0 = torch.as_tensor(init.hidden_init((B, 64, 64, channels), seed=5 + seed_off)).cuda()
        m = mp.model()
        m.channels, m.timesteps, m.compute_mode, m.hidden_state = channels, timesteps, mode, h0
        m.load_params(P)
        return m

    def measure(m, channels, timesteps, mode, B, depth_dev, depth_pin, steps, warmup, with_clocks, gather):
        """W warm-up steps, then K timed steps of the device-resident forward (+ the all-gather of the predictions
        when sharded), the conv kernels timed live; then the same through host buffers."""
        # sharded: every step's predictions are all-gathered, asynchronously into one of two buffers, so a step does
        # not wait for the collective (and through it for the slowest rank) before the next forward starts
        gatherer = PredictionGatherer(B, 69, device="cuda") if (gather and world > 1) else None
        last = [None]

        def step_dev():
            out = m.build(depth_dev, 69)
            last[0] = out
            if gatherer is not None:
                gatherer.submit(out)
                if os.environ.get("BENCH_SYNC_GATHER") == "1":      # A/B switch: wait for every step's collective
                    gatherer.result()
            return out

        def step_host():
            return m.build(depth_pin, 69)          # H2D of the crops + forward + D2H of the predictions

        for _ in range(max(3, warmup)):
            step_dev()
        clocks = Clocks(local) if (with_clocks and rank == 0) else None
        if clocks:
            clocks.wait_ready()
        step_dev()  # the sampler start-up left rank 0's GPU idle: one more untimed step (every rank: it has a collective)
        lib.hgru_enable_kernel_timing(1)
        ms_dev, t0, t1 = timed(step_dev, steps, gatherer.drain if gatherer is not None else None)
        k_ms, k_n = ctypes.c_float(0), ctypes.c_int(0)
        lib.pose_plan_kernel_times(m._plan, ctypes.byref(k_ms), ctypes.byref(k_n))   # last step's hconv launches
        g_mean, g_min = ctypes.c_float(0), ctypes.c_float(0)
        lib.pose_plan_sm_clock_ghz(m._plan, ctypes.byref(g_mean), ctypes.byref(g_min))
        lib.hgru_enable_kernel_timing(0)
        # what the last timed step handed its caller: this rank's predictions, or every rank's once gathered
        last_out = gatherer.result().clone() if gatherer is not None else last[0]
        clk = clocks.stop(t0, t1) if clocks else None
        if clk is not None:
            # nvidia-smi keeps reporting the nominal clock; this is what the conv kernel's own clock64 / %globaltimer saw
            clk["sm_clock_in_kernel_ghz"] = round(float(g_mean.value), 4) if g_mean.value else None
            clk["sm_clock_in_kernel_ghz_min_cta"] = round(float(g_min.value), 4) if g_min.value else None
        launches = m.gpu_launches
        out_check = step_dev()
        if gatherer is not None:
            out_check = gatherer.result().clone()       # [world * B, 69], rank order = batch order
        assert torch.isfinite(out_check).all()
        ms_host = None
        if depth_pin is not None:
            for _ in range(2):
                step_host()
            ms_host, _, _ = timed(step_host, steps)
            # the same host batches as a stream (double-buffered upload / read-back around the forward)
            sf = mp.StreamedForward(m, 69)
            two = [depth_pin, depth_pin.clone().pin_memory()]

            def run_stream(n):
                last = None
                for last in sf(two[i & 1] for i in range(n)):
                    pass
                return last
            run_stream(3)
            ms_stream, _, _ = timed(lambda: run_stream(steps), 1)
            assert torch.equal(run_stream(1), step_host())
        flops_per_launch = 2.0 * B * 64 * 64 * 15 * 15 * channels * channels     # SURVEY 8(d): 2*H*W*S^2*k^2 per frame
        res = {"ms_dev": ms_dev, "ms_host": ms_host, "ms_stream": ms_stream if depth_pin is not None else None,
               "launches_per_step": launches, "clk": clk,
               "flops_per_launch": flops_per_launch, "roof": None, "out": out_check, "last_out": last_out,
               "sm_clock_in_kernel_ghz": round(float(g_mean.value), 4) if g_mean.value else None}
        if k_n.value > 0 and mode in ("bf16", "bf16x3"):
            avg_ms = k_ms.value / k_n.value
            ach = flops_per_launch / (avg_ms * 1e-3) * 1e-12
            kern = ("hconv_tc_kernel SPLIT3 (15x15 implicit GEMM, bf16 hi/lo operand splits = 3 MMAs per useful one, "
                    "tcgen05)" if mode == "bf16x3" else
                    "hconv_stack_kernel (15x15 tap-stacked implicit GEMM + fused gates, tcgen05)" if channels <= 32 else
                    "hconv_tc_kernel FUSE (15x15 implicit GEMM + fused gates, tcgen05)")
            res["roof"] = {"bound": "tensor", "kernel": kern, "achieved": ach, "peak": peak, "unit": "TFLOP/s",
                           "frac": ach / peak, "frac_of_burst": ach / peak_burst, "peak_burst": peak_burst,
                           "peak_source": peak_src, "avg_launch_ms": avg_ms, "launches_per_step": k_n.value,
                           "share_of_step": k_ms.value / (ms_dev / steps), "flops_per_launch": flops_per_launch,
                           "flops_note": "algorithmic, un-padded: 2*N*H*W*S^2*k^2"}
        return res

    B = a.batch
    depth_np = init.synthetic_depth(B, seed=1234 + rank)
    depth_dev = torch.as_tensor(depth_np).cuda()
    depth_pin = torch.as_tensor(depth_np).pin_memory()
    m = make_model(a.channels, a.timesteps, a.mode, B, rank)
    r = measure(m, a.channels, a.timesteps, a.mode, B, depth_dev, depth_pin, a.steps, a.warmup, True, True)

    # sharded run: the gathered predictions are those of the unsharded forward (rank 0 recomputes the last rank's shard)
    shard_check = None
    if world > 1:
        if rank == 0:
            other = world - 1
            d2 = torch.as_tensor(init.synthetic_depth(B, seed=1234 + other)).cuda()
            m.hidden_state = torch.as_tensor(init.hidden_init((B, 64, 64, a.channels), seed=5 + other)).cuda()
            mine = m.build(d2, 69)
            shard_check = "ok" if torch.equal(mine, r["out"][other * B:(other + 1) * B]) else "MISMATCH"
        sync()
    ms_dev, ms_host = r["ms_dev"], r["ms_host"]

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    if a.dump_outputs:
        dump_output(a.dump_outputs, "out_put", r["last_out"].cpu().numpy())
    frames = B * world * a.steps
    value = frames / (ms_dev * 1e-3)
    e2e = frames / (ms_host * 1e-3)
    k = a.channels
    roof = r["roof"]
    if roof is not None:
        traffic, tsrc = None, None
        try:
            tj = json.load(open(os.path.join(ROOT, "profiles", "r02_ncu_traffic.json"))).get(str(k))
            if tj and tj.get("batch") == B and tj.get("timesteps", 8) == a.timesteps:
                traffic, tsrc = tj["bytes_per_launch"], tj.get("source")
        except Exception:
            pass
        roof["traffic"] = traffic
        roof["traffic_source"] = tsrc or "no ncu --set full capture for this configuration"
    cpu = None
    if not a.no_cpu_baseline:
        fps, med, cores = cpu_forward_fps(a, a.cpu_frames, 3)
        cpu = {"value": fps, "unit": UNIT, "cores": cores, "kind": "port",
               "sample": "%d of the %d frames, median of 3 forwards (%.1f s each), torch-CPU oracle "
                         "(stand-in for TF-CPU: TensorFlow absent)" % (a.cpu_frames, B, med)}
    stages = None
    if not a.no_stages and world == 1 and a.mode == "bf16":
        try:
            stages = neighbour_stages(a, m, torch, mp, init)
        except Exception as e:                      # never lose the headline line to an auxiliary measurement
            stages = {"error": repr(e)}
    # The other BASELINE configs on this GPU, short runs (N = 1, default workload only): the reference's own width
    # (64 channels), the deep variant (32 channels, T = 16) and the fp32-class tensor-core arithmetic at 25 channels.
    extra = None
    default_workload = (a.channels, a.timesteps, a.mode, B) == (25, 8, "bf16", 256)
    if world == 1 and default_workload and not a.no_extra:
        extra = {}
        del m
        for key, (ch, T, mode) in (("k64_T8", (64, 8, "bf16")), ("deep_k32_T16", (32, 16, "bf16")),
                                   ("k25_T8_bf16x3", (25, 8, "bf16x3"))):
            try:
                torch.cuda.empty_cache()
                mx = make_model(ch, T, mode, B, 0)
                rx = measure(mx, ch, T, mode, B, depth_dev, None, 3, 3, False, False)
                flops_step = 2 * T * rx["flops_per_launch"]
                extra[key] = {"workload": "batch %d, %d channels, T=%d, %s (%s)" % (B, ch, T, mode, config_label(B, ch, T)),
                              "value": B * 3 / (rx["ms_dev"] * 1e-3), "unit": UNIT, "ms_per_step": rx["ms_dev"] / 3,
                              "steps": 3, "gpu_launches_per_step": rx["launches_per_step"],
                              "hconv_TFLOP/s_whole_step": flops_step / (rx["ms_dev"] / 3 * 1e-3) * 1e-12,
                              "roofline": rx["roof"], "sm_clock_in_kernel_ghz": rx["sm_clock_in_kernel_ghz"]}
                del mx, rx
            except Exception as e:
                extra[key] = {"error": repr(e)}
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": n_gpus, "steps": a.steps,
            "warmup": max(3, a.warmup), "ms_per_step": ms_dev / a.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": a.mode if a.mode != "fp32" else "f32",
            "data": "synthetic", "config": workload_config(a, n_gpus),
            "e2e": {"value": e2e, "unit": UNIT, "h2d_bytes_per_step": int(depth_pin.numel() * 4) * world,
                    "d2h_bytes_per_step": int(B * 69 * 4) * world, "ms_per_step": ms_host / a.steps,
                    "streamed": {"value": frames / (r["ms_stream"] * 1e-3), "unit": UNIT,
                                 "ms_per_step": r["ms_stream"] / a.steps,
                                 "note": "the same host batches through monkey_pose_b200.StreamedForward: upload of "
                                         "batch i+1 and read-back of batch i-1 overlap the forward of batch i (the role "
                                         "of the reference's input queues); `value` above it is the synchronous "
                                         "model.build(host batch) call"}},
            "gpu_launches": int(r["launches_per_step"] * a.steps), "clocks": r["clk"], "roofline": roof,
            "cpu_baseline": cpu, "neighbour_stages": stages, "extra": extra, "shard_check": shard_check,
            "tensor_util_whole_step": (2 * a.timesteps * r["flops_per_launch"] * world * a.steps / (ms_dev * 1e-3)) * 1e-12
            / (peak * world)}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def neighbour_stages(a, m, torch, mp, init_mod):
    """SURVEY 8(f) rows 1 + 2, measured at the same batch on rank 0: the GPU crop stage before the network
    (prepare_data_test -> cropArea3D) and the post-processing after it (absolute coordinates + joint error), plus
    the whole chain camera frames -> joints through the public API with host buffers.  HBM-bound byte work:
    GB/s against MEASURED_PEAKS.json hbm_gbps."""
    import numpy as np
    from monkey_pose_b200 import tf_monkeydetector as tmd
    from monkey_pose_b200 import pose_evaluation as pe

    class Cfg(object):
        image_orig_size = [424, 512, 1]
        image_target_size = [128, 128, 1]
        image_max_depth = 10000.

    B, h, w = a.batch, 424, 512
    rng = np.random.default_rng(99)
    base = np.round(rng.uniform(600, 4000, size=(8, h, w)) / 8) * 8
    base[rng.uniform(size=base.shape) < 0.05] = 0
    frames_np = (base[rng.integers(0, 8, B)] / 10000.0).astype(np.float32)
    coms_norm = np.stack([rng.uniform(0.3, 0.9, B), rng.uniform(0.25, 0.7, B), rng.uniform(0.1, 0.3, B)], 1)
    md = tmd.tfMonkeyDetector(365.456, 365.456, 256, 212, [800, 800, 1200], 200, 10000)
    frames_dev = torch.as_tensor(frames_np).cuda()
    frames_pin = torch.as_tensor(frames_np).pin_memory()
    labels = torch.rand(B, 23, 3, device="cuda") * 100.0

    def ev_time(fn, reps=5):
        fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record()
        for _ in range(reps):
            r = fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps, (time.perf_counter() - t0) * 1e3 / reps, r

    patches, coms, _ = tmd.prepare_data_test(frames_dev, coms_norm, md, Cfg())
    # algorithmic bytes of the crop: every source pixel of each frame's window once + the 128x128 output
    ints, _, _ = md._windows_batch(np.asarray(coms), h, w, (128, 128))
    x0, y0, wb, hb = [ints[:, i].astype(np.int64) for i in range(4)]
    win_px = int((np.clip(np.minimum(x0 + wb, w) - np.maximum(x0, 0), 0, None) *
                  np.clip(np.minimum(y0 + hb, h) - np.maximum(y0, 0), 0, None)).sum())
    crop_bytes = 4.0 * win_px + 4.0 * B * 128 * 128
    crop_gpu_ms, crop_wall_ms, _ = ev_time(lambda: tmd.prepare_data_test(frames_dev, coms_norm, md, Cfg()))
    coms_f32_dev = torch.as_tensor(coms_norm.astype(np.float32)).cuda()
    crop_dev_ms, crop_dev_wall_ms, _ = ev_time(lambda: tmd.prepare_data_test(frames_dev, coms_f32_dev, md, Cfg()))
    # the kernel alone, through the C ABI, parameters already on the device
    lib = mp._lib.load()
    _, zf, _ = md._windows_batch(np.asarray(coms), h, w, (128, 128))
    ip_d, zp_d = torch.as_tensor(ints).cuda(), torch.as_tensor(zf).cuda()
    out_d = torch.empty((B, 128, 128), device="cuda", dtype=torch.float32)
    stream = torch.cuda.current_stream().cuda_stream

    def crop_kernel():
        mp._lib.check(lib.crop_area3d_forward(frames_dev.data_ptr(), B, h, w, 10000.0, ip_d.data_ptr(),
                                              zp_d.data_ptr(), float(md.maxDepth), 10000.0, out_d.data_ptr(),
                                              128, 128, stream), "crop_area3d_forward")

    crop_kernel_ms, _, _ = ev_time(crop_kernel, 20)
    out = m.build(patches, 69)
    post_gpu_ms, post_wall_ms, _ = ev_time(lambda: pe.getMeanError_np(
        labels, md.getAbsoluteCoordinates_batch(out, coms, 600.0)[0]))

    # attention (centre-of-mass) CNN at the reference's widths: the network that produces the crop centres
    am = mp.attn_model_struct()
    am.load_params(init_mod.attn_params(seed=8))
    attn_gpu_ms, attn_wall_ms, attn_out = ev_time(lambda: am.build(frames_dev, 3), 3)
    attn_flops = 2.0 * B * (128 * 128 * 9 * 64 + 64 * 64 * 9 * 64 * 128 + 32 * 32 * 9 * 128 * 256 +
                            16 * 16 * 9 * 256 * 512 + 8 * 8 * 25 * 512 * 1024 + 16384 * 1024 + 1024 * 3)

    coms_norm_dev = torch.as_tensor(coms_norm.astype(np.float32)).cuda()

    def chain():
        f = frames_pin.cuda(non_blocking=True)
        am.build(f, 3)                               # its output would drive the crop; fixed centres keep it valid
        # centres as a device tensor: window arithmetic, crop, network and post-processing without a host round trip
        p, cs, _ = tmd.prepare_data_test(f, coms_norm_dev, md, Cfg())
        xyz, _ = md.getAbsoluteCoordinates_batch(m.build(p, 69), cs, 600.0)
        return xyz.cpu()

    chain_gpu_ms, chain_wall_ms, _ = ev_time(chain, 3)
    # the same chain through the package's pipeline helper: upload in four pieces on a copy stream, the attention CNN
    # on each piece as it lands
    pipe = mp.FramesToJoints(am, m, md, Cfg(), cube_z=1200.0, chunks=4)
    _, pipe_wall_ms, _ = ev_time(lambda: pipe(frames_pin, centres=coms_norm_dev), 3)
    # ... and fed raw 16-bit millimetre frames (what a depth camera delivers; thresholds + normalisation on the device)
    raw_pin = torch.from_numpy(np.round(frames_np * 10000.0).astype(np.uint16).view(np.int16)).pin_memory()
    _, pipe16_wall_ms, _ = ev_time(lambda: pipe(raw_pin, centres=coms_norm_dev), 3)
    hbm = None
    try:
        hbm = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))).get("hbm_gbs")
    except Exception:
        pass
    # the centre-of-mass estimate the crop stage falls back to without an attention output (calculateCoM on every
    # frame, numpy's float32 summation order reproduced): one read of every frame, HBM-bound
    try:
        def ev_best(fn, reps=10):
            # a dozen short launches per call: the host's launch gaps are inside any event interval, so take the
            # best of `reps` single calls instead of their mean
            fn()
            fn()
            torch.cuda.synchronize()
            best = float("inf")
            for _ in range(reps):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                fn()
                e1.record()
                torch.cuda.synchronize()
                best = min(best, e0.elapsed_time(e1))
            return best

        com_ms = ev_best(lambda: md.calculateCoM_batch(frames_dev, frame_scale=10000.0))
        docom_ms = ev_best(lambda: md.cropArea3D_batch_device(frames_dev, frame_scale=10000.0, out_divisor=10000.0,
                                                              docom=True))
        com_gbs = 4.0 * B * h * w / (com_ms * 1e-3) * 1e-9
        com_stage = {"calculate_com_ms": com_ms, "algorithmic_bytes": 4.0 * B * h * w, "GB/s": com_gbs,
                     "frac_of_hbm": (com_gbs / hbm) if hbm else None, "crop_with_estimated_and_refined_com_ms": docom_ms,
                     "note": "best of 10 single calls; calculate_com_forward (2 kernels + a 8 KB memset) on 424x512 frames resident in HBM; "
                             "second figure: cropArea3D(com=None, docom=True) for the batch = CoM of the frame, "
                             "window, CoM of the window, window, crop"}
    except Exception as e:
        com_stage = {"error": repr(e)}
    crop_gbs = crop_bytes / (crop_kernel_ms * 1e-3) * 1e-9
    return {"batch": B, "frame": [h, w],
            "crop": {"kernel_ms": crop_kernel_ms, "algorithmic_bytes": crop_bytes, "GB/s": crop_gbs,
                     "frac_of_hbm": (crop_gbs / hbm) if hbm else None,
                     "api_ms": crop_gpu_ms, "api_wall_ms": crop_wall_ms,
                     "api_device_windows_ms": crop_dev_ms, "api_device_windows_wall_ms": crop_dev_wall_ms,
                     "note": "kernel_ms: crop_area3d_forward alone (C ABI, parameters on the device); api_ms: "
                             "prepare_data_test = host window arithmetic (comToBounds) + parameter upload + "
                             "kernel; api_device_windows_ms: the same with the centres of mass as a CUDA tensor "
                             "(crop_windows_forward + crop_area3d_forward, no host round trip); frames resident in HBM"},
            "com_estimate": com_stage,
            "post": {"gpu_ms": post_gpu_ms, "wall_ms": post_wall_ms,
                     "note": "x600 + CoM, xyz->uvd, mean joint error; 23 joints per frame, latency-bound"},
            "attention_cnn": {"gpu_ms": attn_gpu_ms, "frames_per_s": B / (attn_gpu_ms * 1e-3),
                              "algorithmic_TFLOP/s": attn_flops / (attn_gpu_ms * 1e-3) * 1e-12,
                              "launches": am.gpu_launches,
                              "note": "attn_model_struct.build at 64..1024 channels: resize + 5 x (conv, relu, "
                                      "pool, batch-norm) + 2 fc; convs 2-5 as implicit tcgen05 GEMMs (4-D TMA boxes of the NHWC "
                                      "activation per tap) with bf16 hi/lo splits (3 MMAs per k-step)"},
            "frames_to_joints_pipelined_e2e": {"value": B / (pipe_wall_ms * 1e-3), "unit": UNIT, "wall_ms": pipe_wall_ms,
                                               "note": "monkey_pose_b200.FramesToJoints: same stages, upload in 4 pieces "
                                                       "on a copy stream under the attention CNN"},
            "frames_to_joints_pipelined_raw16_e2e": {"value": B / (pipe16_wall_ms * 1e-3), "unit": UNIT,
                                                     "wall_ms": pipe16_wall_ms, "h2d_bytes": int(raw_pin.numel() * 2),
                                                     "note": "the same fed raw 16-bit depth (mm): half the upload"},
            "frames_to_joints_e2e": {"value": B / (chain_wall_ms * 1e-3), "unit": UNIT, "wall_ms": chain_wall_ms,
                                     "stages": "H2D frames, attention CNN, crop, hGRU pose net, post-processing, "
                                               "D2H joints",
                                     "h2d_bytes": int(frames_np.nbytes), "d2h_bytes": int(B * 69 * 4)}}


def main():
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)


if __name__ == "__main__":
    main()
