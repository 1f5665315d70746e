"""GPU (B200): the attention CNN's fp16 compute mode (attn_model_struct.compute_mode = 'fp16', HGRU_MODE_FP16 of
attn_plan_create_mode): fp16 GEMM operands for aconv_2 .. aconv_5 and afc_1, one tcgen05 product per k-step, fp32
accumulation.  Every activation within 2.5e-3 of the fp64 oracle, the batch-capacity rule, saturation, the bf16x3
mode of the new entry point, and the camera-frames -> joints pipeline driven by an fp16 attention CNN."""
import ctypes
import os

import numpy as np
import pytest
import torch

import monkey_pose_b200 as mp
from monkey_pose_b200 import _lib
from monkey_pose_b200 import initialization as init
from oracle import attn_oracle_torch as atorch
from oracle import hgru_oracle_np as onp

pytestmark = pytest.mark.gpu

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "attn_ref.npz")
TOL = 2.5e-3
NAMES = ("resized", "pool1", "pool2", "pool3", "pool4", "pool5", "fc1")
REF_WIDTHS = (64, 128, 256, 512, 1024)


def _st():
    return torch.cuda.current_stream().cuda_stream


def _model(P, mode, widths=REF_WIDTHS, fc=1024):
    am = mp.attn_model_struct()
    am.widths, am.fc_hidden, am.compute_mode = widths, fc, mode
    am.load_params(P)
    return am


def _frames(n, h, w, seed):
    rng = np.random.default_rng(seed)
    f = rng.uniform(0.06, 0.4, size=(n, h, w, 1)).astype(np.float32)
    f[rng.uniform(size=f.shape) < 0.05] = 0.0
    return f


def _golden():
    z = np.load(GOLDEN)
    return z["frames"], {k[4:]: z[k] for k in z.files if k.startswith("var:")}


def _case(name):
    if name == "golden":                     # widths 8..32: every conv on the explicit im2col path
        frames, P = _golden()
        return frames, P, tuple(int(P["%s/%s_filters" % (c, c)].shape[3]) for c, _ in init.ATTN_CONV), 1024
    if name == "reference-widths":           # Cin % 64 == 0: convs 2..5 as implicit GEMMs, afc_1 explicit
        return _frames(16, 424, 512, 3), init.attn_params(REF_WIDTHS, 1024, 3, seed=5, random_bn=True), REF_WIDTHS, 1024
    widths = (8, 24, 16, 40, 32)             # small odd widths: explicit im2col with padded K
    return _frames(5, 96, 80, 4), init.attn_params(widths, 64, 3, seed=6, random_bn=True), widths, 64


@pytest.mark.parametrize("case", ["golden", "reference-widths", "small-widths"])
def test_fp16_every_activation_within_bar_of_fp64_oracle(case):
    frames, P, widths, fc = _case(case)
    am = _model(P, "fp16", widths, fc)
    out = am.build(torch.as_tensor(frames).cuda(), 3)
    ref, acts = atorch.attn_forward(frames, P, dtype=torch.float64, trace=True)
    acts = {k: v.numpy() for k, v in acts.items()}
    acts["resized"] = atorch.resize_bilinear_tf1(frames, 128, 128)
    for name in NAMES:
        got = am.activation(name).cpu().numpy()
        want = acts[name].reshape(got.shape)
        err = onp.rel_err(got, want)[0]
        assert err < TOL, (name, err)
    err = onp.rel_err(out.cpu().numpy(), ref.numpy())[0]
    assert err < TOL, ("out_put", err)
    assert torch.equal(out, am.build(torch.as_tensor(frames).cuda(), 3))           # deterministic


def test_create_mode_bf16x3_equals_attn_plan_create_bitwise(monkeypatch):
    """A bf16x3 plan from attn_plan_create_mode is attn_plan_create's plan: the same output, activations and
    launches."""
    frames = torch.as_tensor(_frames(6, 212, 256, 7)).cuda()
    P = init.attn_params(REF_WIDTHS, 1024, 3, seed=5, random_bn=True)
    lib = _lib.load()
    a = _model(P, "bf16x3")
    out_a = a.build(frames, 3)
    acts_a = {n: a.activation(n) for n in NAMES}
    create_mode = lib.attn_plan_create_mode
    monkeypatch.setattr(lib, "attn_plan_create", lambda N, H, W, w, F, O, out: create_mode(
        N, H, W, w, F, O, _lib.MODE_BF16X3, out))
    b = _model(P, "bf16x3")
    out_b = b.build(frames, 3)
    torch.cuda.synchronize()
    assert torch.equal(out_a, out_b)
    for n in NAMES:
        assert torch.equal(acts_a[n], b.activation(n)), n
    assert a.gpu_launches == b.gpu_launches
    assert lib.attn_plan_workspace_bytes(a._plan) == lib.attn_plan_workspace_bytes(b._plan)


def test_fp16_plan_holds_no_lo_halves():
    frames = torch.as_tensor(_frames(3, 96, 128, 8)).cuda()
    P = init.attn_params(REF_WIDTHS, 1024, 3, seed=5)
    lib = _lib.load()
    ws = {}
    for mode in ("bf16x3", "fp16"):
        am = _model(P, mode)
        am.build(frames, 3)
        ws[mode] = lib.attn_plan_workspace_bytes(am._plan)
    # weights alone: afc_1 16384 x 1024 and the conv filters, 2 bytes per lo value
    lo_weights = 2 * (16 * 1024 * 1024 + 9 * 64 * 128 + 9 * 128 * 256 + 9 * 256 * 512 + 25 * 512 * 1024)
    assert ws["bf16x3"] - ws["fp16"] >= lo_weights, ws


@pytest.mark.parametrize("widths", [(64, 64, 64, 64, 64), REF_WIDTHS, (8, 24, 16, 40, 32)])
def test_fp16_forward_batch_equals_dedicated_plan(widths):
    """Odd n on a capacity-7 fp16 plan: bitwise the plan created for n frames, the same launches."""
    cap, fc = 7, 64
    lib = _lib.load()
    frames = torch.rand(cap, 120, 160, device="cuda", generator=torch.Generator("cuda").manual_seed(3))
    P = init.attn_params(widths=widths, fc_hidden=fc, out=3, seed=8, random_bn=True)
    big = _model(P, "fp16", widths, fc)
    big.build(frames, 3)
    for n in (1, 3, 5, 7):
        ded = _model(P, "fp16", widths, fc)
        want = ded.build(frames[:n].contiguous(), 3)
        want_acts = {name: ded.activation(name).reshape(-1) for name in NAMES}
        out = torch.full((n, 3), float("nan"), device="cuda")
        _lib.check(lib.attn_forward_batch(big._plan, n, frames.data_ptr(), out.data_ptr(), _st()),
                   "attn_forward_batch")
        acts = {}
        for name in NAMES:
            dst = torch.full((want_acts[name].numel() + 16,), float("nan"), device="cuda")
            _lib.check(lib.attn_get_activation(big._plan, name.encode(), dst.data_ptr(), _st()), "attn_get_activation")
            acts[name] = dst
        torch.cuda.synchronize()
        assert torch.equal(out, want), n
        assert lib.attn_plan_launch_count(big._plan) == lib.attn_plan_launch_count(ded._plan)
        for name, a in acts.items():
            b = want_acts[name]
            assert torch.equal(a[:b.numel()], b), (n, name)
            assert torch.isnan(a[b.numel():]).all(), (n, name)


@pytest.mark.parametrize("widths", [REF_WIDTHS, (8, 24, 16, 40, 32)])
def test_fp16_saturating_inputs_stay_finite(widths):
    """Activations and weights beyond fp16's +-65504 are clamped by the operand conversions, never inf / NaN."""
    P = init.attn_params(widths=widths, fc_hidden=64, out=3, seed=9)
    P = dict(P)
    P["aconv_3/aconv_3_filters"] = P["aconv_3/aconv_3_filters"] * np.float32(1e5)
    P["afc_1/afc_1_weights"] = P["afc_1/afc_1_weights"] * np.float32(1e5)
    frames = torch.as_tensor(_frames(3, 96, 128, 10) * np.float32(1e6)).cuda()
    am = _model(P, "fp16", widths, 64)
    out = am.build(frames, 3)
    torch.cuda.synchronize()
    assert am.activation("pool1").abs().max().item() > 65504           # the GEMM operands did saturate
    assert torch.isfinite(out).all()
    for name in NAMES:
        assert torch.isfinite(am.activation(name)).all(), name


class _Cfg(object):
    image_orig_size = [424, 512, 1]
    image_target_size = [128, 128, 1]
    image_max_depth = 10000.


def _scenes(n, h, w, seed):
    """n distinct depth frames / 10 m: an ellipsoidal object at a random place and depth in front of a noisy wall"""
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:h, 0:w].astype(np.float32)
    out = np.empty((n, h, w), np.float32)
    for i in range(n):
        f = rng.uniform(3200, 4000) + rng.normal(0, 20, (h, w))
        cy, cx, d = rng.uniform(0.2, 0.8) * h, rng.uniform(0.2, 0.8) * w, rng.uniform(1200, 2800)
        r2 = ((yy - cy) / rng.uniform(40, 90)) ** 2 + ((xx - cx) / rng.uniform(30, 70)) ** 2
        f = np.where(r2 < 1, d - 150 * np.sqrt(np.clip(1 - r2, 0, 1)), f)
        f[rng.uniform(size=(h, w)) < 0.05] = 0
        out[i] = np.round(f) / 10000.0
    return out


def test_frames_to_joints_with_an_fp16_attention_cnn():
    """FramesToJoints driven by the attention output (no fixed centres): finite joints, every frame's crop window
    valid whenever the bf16x3 pipeline's is, and fp16 centres within 4 px / 12 mm of bf16x3's (a window is ~146 px
    wide at 2 m).  afc_out is calibrated on the bf16x3 forward so that the centres spread over the frame like a
    trained head's (standard deviation 0.12 of the height / width, 300 mm); the fp16 error at the output grows with
    that spread."""
    from monkey_pose_b200 import tf_monkeydetector as tmd
    n, h, w = 16, 424, 512
    frames_np = _scenes(n, h, w, 21)
    f_dev = torch.as_tensor(frames_np).cuda()
    P = dict(init.attn_params(REF_WIDTHS, 1024, 3, seed=8))
    P["afc_out/afc_out_biases"] = np.zeros(3, np.float32)
    raw = _model(P, "bf16x3").build(f_dev, 3).double().cpu().numpy()
    scale = np.array([0.12, 0.12, 0.03]) / raw.std(axis=0)
    P["afc_out/afc_out_weights"] = (P["afc_out/afc_out_weights"] * scale).astype(np.float32)
    P["afc_out/afc_out_biases"] = (np.array([0.5, 0.5, 0.2]) - scale * raw.mean(axis=0)).astype(np.float32)
    pm = mp.model()
    pm.channels, pm.timesteps, pm.fc_hidden = 25, 2, 32
    pm.hidden_state = init.hidden_init((n, 64, 64, 25), seed=5)
    pm.load_params(init.pose_params(channels=25, S=15, T=2, hw=64, fc_hidden=32, out=69, seed=3, stress=4.0))
    res = {}
    for mode in ("bf16x3", "fp16"):
        md = tmd.tfMonkeyDetector(365.456, 365.456, 256, 212, [800, 800, 1200], 200, 10000)
        am = _model(P, mode)
        pipe = mp.FramesToJoints(am, pm, md, _Cfg(), cube_z=1200.0, chunks=4)
        xyz, uvd = pipe(torch.as_tensor(frames_np).pin_memory())
        res[mode] = (xyz, uvd, md.last_invalid_dev.cpu().numpy(), pipe._tr.double().cpu().numpy())
    xyz, uvd, inv16, tr16 = res["fp16"]
    _, _, inv3, tr3 = res["bf16x3"]
    assert xyz.shape == (n, 23, 3) and torch.isfinite(xyz).all() and torch.isfinite(uvd).all()
    assert tr3[:, 0].std() * h > 25 and tr3[:, 1].std() * w > 25, tr3     # the centres do move over the frame
    assert (inv3 == 0).all(), inv3
    assert not np.any((inv3 == 0) & (inv16 != 0)), (inv3, inv16)
    assert (np.abs(tr16 - tr3).max(axis=0) * np.array([h, w, 10000.0]) <= [4.0, 4.0, 12.0]).all(), (tr16 - tr3)
