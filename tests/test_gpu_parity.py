"""GPU (B200): the CUDA path, called through the C-ABI by the reference-shaped Python classes,
against the oracle -- golden fixtures produced by the reference source, seeded random cases, edge
shapes, and size-independent properties at BASELINE sizes.

Tolerances (BASELINE.json north_star): fp32 path <= 1e-4 relative on hidden states and outputs;
bf16 tensor-core path <= 1e-2 relative and <= 0.5 mm mean per-joint deviation."""
import glob
import os

import numpy as np
import pytest
import torch

import monkey_pose_b200 as mp
from monkey_pose_b200 import initialization as init
from oracle import hgru_oracle_np as onp
from oracle import hgru_oracle_torch as otorch

pytestmark = pytest.mark.gpu

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
HGRU_FILES = sorted(glob.glob(os.path.join(GOLDEN, "hgru_ref_*.npz")))
POSE_AUX = mp.model().aux
TOL = {"fp32": 1e-4, "bf16": 1e-2, "bf16x3": 1e-4}


def _run_cc(X, O0, params, T, S, mode, trace=True):
    cc = mp.ContextualCircuit(X=torch.as_tensor(X).cuda(), timesteps=T, SRF=1, SSN=S, SSF=S, aux=POSE_AUX,
                              params=params, hidden_state=O0, compute_mode=mode)
    O, weights, acts = cc.build(trace=trace)
    torch.cuda.synchronize()
    return cc, O, weights


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
@pytest.mark.parametrize("path", HGRU_FILES, ids=[os.path.basename(p) for p in HGRU_FILES])
def test_hgru_matches_reference_golden_every_timestep(path, mode):
    z = np.load(path)
    T, S = int(z["T"]), int(z["S"])
    params = {n: z["var:contextual_circuit/" + n] for n in onp.HGRU_PARAM_NAMES}
    cc, O, weights = _run_cc(z["X"], z["O0"], params, T, S, mode)
    for t in range(T):
        e1 = onp.rel_err(cc.I_steps[t].cpu().numpy(), z["I_steps"][:, t])[0]
        e2 = onp.rel_err(cc.O_steps[t].cpu().numpy(), z["O_steps"][:, t])[0]
        assert e1 < TOL[mode] and e2 < TOL[mode], (t, e1, e2)
    assert onp.rel_err(O.cpu().numpy(), z["O_final"])[0] < TOL[mode]
    assert set(weights.keys()) == set(z["weights_keys"].tolist())
    assert cc.gpu_launches > 0


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
@pytest.mark.parametrize("shape", [(1, 64, 64, 64, 15, 2), (2, 64, 64, 25, 15, 2), (1, 20, 36, 32, 15, 2),
                                   (3, 16, 16, 16, 5, 3), (1, 7, 9, 3, 3, 2),
                                   # remainder-packed k <= 25 kernel: ragged H/W, two x-units per row (W > 64),
                                   # k = 24 / 17 (the row-packed 25th-channel plane is all zero), T = 3
                                   (2, 40, 24, 25, 15, 3), (1, 33, 70, 25, 15, 2), (1, 18, 66, 24, 15, 2),
                                   (1, 64, 64, 17, 15, 2),
                                   # 33..48 channels are padded to 64 on the tensor-core paths
                                   (2, 19, 21, 48, 15, 2),
                                   # 64 channels (paired-tap schedule), ragged: the second 32-pixel unit of a row and
                                   # the third 16-row unit of a frame are partly outside the image
                                   (1, 37, 45, 64, 15, 2)])
def test_hgru_seeded_cases_vs_oracle(shape, mode):
    """k = 64 (reference), 25 and 32 (BASELINE sweep), ragged H/W, tiny shapes; stress weights so
    tanh leaves its linear region."""
    n, h, w, k, S, T = shape
    rng = np.random.default_rng(5)
    X = rng.uniform(-1, 1, size=(n, h, w, k)).astype(np.float32)
    O0 = init.hidden_init((n, h, w, k), seed=3, limit=0.5)
    params = init.hgru_params(k, S, T, seed=9, stress=6.0)
    cc, O, _ = _run_cc(X, O0, params, T, S, mode)
    ref, H1s, H2s = otorch.hgru_forward(X, O0, params, T, dtype=torch.float64, trace=True)
    for t in range(T):
        assert onp.rel_err(cc.I_steps[t].cpu().numpy(), H1s[t].numpy())[0] < TOL[mode]
        assert onp.rel_err(cc.O_steps[t].cpu().numpy(), H2s[t].numpy())[0] < TOL[mode]
    assert np.abs(ref.numpy()).max() > 0.05
    assert onp.rel_err(O.cpu().numpy(), ref.numpy())[0] < TOL[mode]


def test_hgru_hidden_init_variants_and_return_convention():
    X = torch.rand(1, 16, 16, 16, device="cuda")
    aux = dict(POSE_AUX, hidden_init="zeros", return_weights=False)
    O = mp.ContextualCircuit(X=X, timesteps=2, SSN=5, SSF=5, aux=aux, compute_mode="fp32").build()
    assert torch.is_tensor(O) and O.shape == X.shape
    params = init.hgru_params(16, 5, 2, seed=42)
    ref = otorch.hgru_forward(X.cpu().numpy(), np.zeros((1, 16, 16, 16), np.float32), params, 2, dtype=torch.float64)
    assert onp.rel_err(O.cpu().numpy(), ref.numpy())[0] < 1e-4
    aux["hidden_init"] = "identity"
    O2 = mp.ContextualCircuit(X=X, timesteps=2, SSN=5, SSF=5, aux=aux, compute_mode="fp32").build()
    ref2 = otorch.hgru_forward(X.cpu().numpy(), X.cpu().numpy(), params, 2, dtype=torch.float64)
    assert onp.rel_err(O2.cpu().numpy(), ref2.numpy())[0] < 1e-4
    aux["hidden_init"] = "bogus"
    with pytest.raises(RuntimeError):
        mp.ContextualCircuit(X=X, timesteps=2, SSN=5, SSF=5, aux=aux).build()


def _pose(mode, N, channels, hw, T, S, fc_hidden, seed=3, stress=4.0, host=False):
    P = init.pose_params(channels=channels, S=S, T=T, hw=hw, fc_hidden=fc_hidden, out=69, seed=seed,
                         stress=stress, random_bn=True)
    depth = init.synthetic_depth(N, seed=0, size=2 * hw)
    h0 = init.hidden_init((N, hw, hw, channels), seed=5)
    m = mp.model()
    m.channels, m.timesteps, m.SSF, m.SSN, m.fc_hidden, m.compute_mode = channels, T, S, S, fc_hidden, mode
    m.hidden_state = h0
    m.load_params(P)
    d = torch.as_tensor(depth)
    out = m.build(d.pin_memory() if host else d.cuda(), 69)
    torch.cuda.synchronize()
    return m, out, P, depth, h0


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
@pytest.mark.parametrize("cfg", [(2, 8, 8, 3, 5, 32), (2, 25, 16, 2, 15, 64), (1, 64, 64, 2, 15, 128)])
def test_pose_model_vs_oracle(cfg, mode):
    N, ch, hw, T, S, F = cfg
    m, out, P, depth, h0 = _pose(mode, N, ch, hw, T, S, F)
    ref, acts = otorch.pose_forward(depth, P, h0, timesteps=T, dtype=torch.float64, trace=True)
    tol = TOL[mode]
    assert onp.rel_err(m.activation("conv3").cpu().numpy(), acts["conv3"].numpy())[0] < tol
    assert onp.rel_err(m.activation("hgru").cpu().numpy(), acts["hgru"].numpy())[0] < tol
    assert onp.rel_err(m.activation("fc1").cpu().numpy(), acts["fc1"].numpy())[0] < tol
    assert onp.rel_err(out.cpu().numpy(), ref.numpy())[0] < tol
    assert onp.mean_joint_error_mm(out.cpu().numpy(), ref.numpy()) < 0.5
    assert out.shape == (N, 69) and m.out_put is out and m.gpu_launches > 0
    assert ("conv_1", 0) in m.var_dict and ("fc_out", 1) in m.var_dict


def test_pose_model_matches_reference_layer_golden():
    """conv_layer / max_pool through the fused stem, against the reference's own layer outputs."""
    z = np.load(os.path.join(GOLDEN, "pose_layers_ref.npz"))
    # stem head only: conv_1 (1->6) + relu + pool, identity batch-norm => compare with pool1
    m = mp.model()
    m.channels, m.timesteps, m.SSF, m.fc_hidden, m.compute_mode = 6, 1, 3, 10, "fp32"
    P = init.pose_params(channels=6, S=3, T=1, hw=6, fc_hidden=10, out=5, seed=1)
    for n in ("conv_1/conv_1_filters", "conv_1/conv_1_biases", "conv_2/conv_2_filters", "conv_2/conv_2_biases"):
        P[n] = z["var:" + n]
    m.load_params(P)
    m.build(torch.as_tensor(z["x"]).cuda(), 5)
    eps_scale = 1.0 / np.sqrt(1.0 + 1e-5)
    assert onp.rel_err(m.activation("pool1").cpu().numpy(), z["pool1"] * eps_scale)[0] < 1e-5
    assert onp.rel_err(m.activation("conv2").cpu().numpy(),
                       onp.conv_layer(z["pool1"] * eps_scale, z["var:conv_2/conv_2_filters"],
                                      z["var:conv_2/conv_2_biases"]) * eps_scale)[0] < 1e-5


def test_stem_activations_on_the_tensor_core_path():
    """bf16 modes keep pool1 / conv2 only as bf16 hi | lo operand copies; `activation()` rebuilds the fp32 tensors
    from them (16 mantissa bits).  Odd width and 25 channels: ragged 4-pixel groups and a padded chunk."""
    outs = {}
    for mode in ("fp32", "bf16"):
        m = mp.model()
        m.channels, m.timesteps, m.fc_hidden, m.compute_mode = 25, 1, 16, mode
        P = init.pose_params(channels=25, S=15, T=1, hw=9, fc_hidden=16, out=5, seed=11, random_bn=True)
        m.load_params(P)
        m.build(torch.as_tensor(init.synthetic_depth(3, seed=4, size=18)).cuda(), 5)
        outs[mode] = {k: m.activation(k).cpu().numpy() for k in ("pool1", "conv2", "conv3")}
    assert onp.rel_err(outs["bf16"]["pool1"], outs["fp32"]["pool1"])[0] < 2e-5
    assert onp.rel_err(outs["bf16"]["conv2"], outs["fp32"]["conv2"])[0] < 1e-4
    assert onp.rel_err(outs["bf16"]["conv3"], outs["fp32"]["conv3"])[0] < 1e-4


def test_chained_launches_equal_stream_ordered_launches(monkeypatch):
    """The stacked conv launches of a forward are chained through per-frame counters (programmatic dependent launch:
    launch l+1 starts while launch l is still running).  Same results, bit for bit, as plain stream order
    (HGRU_NO_CHAIN=1), on every repetition; 150 frames = 600 units on 148 CTAs: several rounds, ragged tail."""
    N, ch, hw, T, S, F = 150, 25, 64, 4, 15, 32
    P = init.pose_params(channels=ch, S=S, T=T, hw=hw, fc_hidden=F, out=69, seed=3, stress=4.0, random_bn=True)
    depth = torch.as_tensor(init.synthetic_depth(N, seed=0, size=2 * hw)).cuda()
    h0 = init.hidden_init((N, hw, hw, ch), seed=5)
    outs = {}
    for chained in (False, True):
        if chained:
            monkeypatch.delenv("HGRU_NO_CHAIN", raising=False)
        else:
            monkeypatch.setenv("HGRU_NO_CHAIN", "1")      # read when the plan is created
        m = mp.model()
        m.channels, m.timesteps, m.fc_hidden, m.compute_mode, m.hidden_state = ch, T, F, "bf16", h0
        m.load_params(P)
        reps = []
        for _ in range(12 if chained else 2):
            reps.append(m.build(depth, 69).clone())
        torch.cuda.synchronize()
        hg = m.activation("hgru")
        for r in reps[1:]:
            assert torch.equal(r, reps[0])
        outs[chained] = (reps[0], hg)
    assert torch.equal(outs[True][0], outs[False][0])
    assert torch.equal(outs[True][1], outs[False][1])


@pytest.mark.parametrize("shape", [(5, 40, 24, 25, 15, 3), (3, 33, 70, 25, 15, 2), (40, 64, 64, 32, 15, 3),
                                   (9, 18, 66, 16, 15, 2)])
def test_chained_layer_equals_traced_layer_on_ragged_shapes(shape):
    """`build(trace=True)` runs the launches in plain stream order (trace copies sit between them); without the
    trace they are chained.  Ragged H / W, two x-units per row, k = 16 / 25 / 32, more units than CTAs: the final
    state must be bitwise the same, and within tolerance of the oracle."""
    n, h, w, k, S, T = shape
    rng = np.random.default_rng(5)
    X = rng.uniform(-1, 1, size=(n, h, w, k)).astype(np.float32)
    O0 = init.hidden_init((n, h, w, k), seed=3, limit=0.5)
    params = init.hgru_params(k, S, T, seed=9, stress=6.0)
    _, O_traced, _ = _run_cc(X, O0, params, T, S, "bf16", trace=True)
    for _ in range(3):
        _, O_chained, _ = _run_cc(X, O0, params, T, S, "bf16", trace=False)
        assert torch.equal(O_chained, O_traced)
    ref = otorch.hgru_forward(X[:2], O0[:2], params, T, dtype=torch.float64)
    ref = ref[0] if isinstance(ref, tuple) else ref
    assert onp.rel_err(O_chained[:2].cpu().numpy(), ref.numpy())[0] < TOL["bf16"]


@pytest.mark.parametrize("N,mode", [(2, "bf16"), (19, "bf16"), (75, "bf16"), (107, "bf16x3"), (75, "fp32")])
def test_pose_host_entry_point_equals_device_entry_point(N, mode):
    """Host buffers in / out (N >= 64: the crops go up in chunks of >= 32 frames, ragged here, and the stem follows
    chunk by chunk) against the device-tensor entry point."""
    m1, out_dev, *_ = _pose(mode, N, 16, 16, 2, 15, 64, host=False)
    m2, out_host, *_ = _pose(mode, N, 16, 16, 2, 15, 64, host=True)
    assert not out_host.is_cuda
    assert torch.equal(out_dev.cpu(), out_host)
    assert torch.equal(m1.activation("conv3"), m2.activation("conv3"))


def test_properties_at_baseline_size_bf16():
    """N = 256, k = 25, T = 8, 15x15 (BASELINE configs[1]): (i) frames are independent -- a frame's
    output does not depend on its batch neighbours (the sharding premise); (ii) determinism;
    (iii) the fp32 and bf16 paths agree within the bf16 budget on a sub-batch."""
    N, ch, hw, T, S, F = 256, 25, 64, 8, 15, 1024
    P = init.pose_params(channels=ch, S=S, T=T, hw=hw, fc_hidden=F, out=69, seed=3)
    depth = init.synthetic_depth(N, seed=1234, size=128)
    h0 = init.hidden_init((N, hw, hw, ch), seed=5)

    def run(mode, sl):
        m = mp.model()
        m.channels, m.compute_mode, m.hidden_state = ch, mode, h0[sl]
        m.load_params(P)
        o = m.build(torch.as_tensor(depth[sl]).cuda(), 69)
        torch.cuda.synchronize()
        return o.cpu().numpy()

    full = run("bf16", slice(0, N))
    again = run("bf16", slice(0, N))
    assert np.array_equal(full, again)
    part = run("bf16", slice(100, 104))
    assert np.array_equal(full[100:104], part)
    exact = run("fp32", slice(100, 104))
    assert onp.rel_err(part, exact)[0] < 1e-2
    assert onp.mean_joint_error_mm(part, exact) < 0.5
    assert np.isfinite(full).all() and np.abs(full).max() > 0


# ---- crop stage (SURVEY 8f rank 1) ------------------------------------------------------------------
class _Cfg(object):
    image_orig_size = [424, 512, 1]
    image_target_size = [128, 128, 1]
    image_max_depth = 10000.


def test_crop_stage_bit_exact_against_reference_golden():
    from monkey_pose_b200 import tf_monkeydetector as tmd
    z = np.load(os.path.join(GOLDEN, "crop_ref.npz"))
    md = tmd.tfMonkeyDetector(365.456, 365.456, 256, 212, [800, 800, 1200], 200, 10000)
    patches, coms, Ms = tmd.prepare_data_test(torch.as_tensor(z["frames"]).cuda(), z["coms_norm"], md, _Cfg())
    torch.cuda.synchronize()
    assert patches.shape == (5, 128, 128, 1)
    assert np.array_equal(patches.cpu().numpy(), z["patches"])           # bit-exact (index + byte work)
    for i in range(5):
        np.testing.assert_allclose(np.asarray(Ms[i]), z["M"][i], rtol=0, atol=1e-12)
        np.testing.assert_allclose(coms[i], z["coms_out"][i], rtol=0, atol=0)
    # no centre of mass given: estimated from the frame (tests/test_gpu_neighbours.py); an empty frame has none -- the
    # reference divides by a zero depth there and fails on int(nan); here the window is flagged and the call raises
    with pytest.raises(ValueError):
        md.cropArea3D(torch.zeros(424, 512, device="cuda"), com=None)
    # a centre of mass whose window misses the frame: that frame becomes an all-background patch, its neighbours are
    # untouched (one wild attention prediction must not abort the batch); the single-frame call raises
    two = torch.as_tensor(z["frames"][:2]).cuda() * 10000.0
    good = z["coms_out"][1]
    out, _, _ = md.cropArea3D_batch(two, [np.array([-900.0, 100.0, 1500.0]), good])
    assert list(md.last_invalid) == [0]
    assert torch.all(out[0] == float(md.maxDepth))
    ref1, _, _ = md.cropArea3D_batch(two[1:], [good])
    assert torch.equal(out[1], ref1[0]) and len(md.last_invalid) == 0
    with pytest.raises(ValueError):
        md.cropArea3D(two[0], com=np.array([-900.0, 100.0, 1500.0]))


def test_crop_stage_vs_oracle_at_batch_size_and_feeds_the_model():
    """256 random frames: the kernel equals the oracle bit for bit, and its output drives model.build."""
    from monkey_pose_b200 import tf_monkeydetector as tmd
    from oracle import crop_oracle_np as crop
    rng = np.random.default_rng(5)
    n, h, w = 256, 424, 512
    base = np.round(rng.uniform(600, 4000, size=(8, h, w)) / 8) * 8
    base[rng.uniform(size=base.shape) < 0.05] = 0
    frames = (base[rng.integers(0, 8, n)] / 10000.0).astype(np.float32)
    # attention outputs: the caller rescales by (height, width, max depth), component 0 is read as x
    coms_norm = np.stack([rng.uniform(0.1, 1.1, n), rng.uniform(0.1, 0.75, n), rng.uniform(0.08, 0.35, n)], 1)
    md = tmd.tfMonkeyDetector(365.456, 365.456, 256, 212, [800, 800, 1200], 200, 10000)
    patches, coms, Ms = tmd.prepare_data_test(torch.as_tensor(frames).cuda(), coms_norm, md, _Cfg())
    ref, _, refM = crop.prepare_data_test(frames, coms_norm, (365.456, 365.456, 256, 212), [800, 800, 1200])
    assert np.array_equal(patches.cpu().numpy(), ref.astype(np.float32))
    np.testing.assert_allclose(np.asarray(Ms[17]), refM[17], rtol=0, atol=1e-12)
    m = mp.model()
    m.channels, m.timesteps, m.fc_hidden = 16, 1, 32
    out = m.build(patches[:4].contiguous(), 69)
    assert out.shape == (4, 69) and torch.isfinite(out).all()


def test_crop_window_arithmetic_on_the_device_equals_the_host():
    """prepare_data_test with the attention outputs as a CUDA tensor: comToBounds + the resize / paste integers + the
    joint transform are computed by crop_windows_forward.  Same patches, centres, matrices and invalid flags as the
    host (numpy float64) path, bit for bit -- including centres whose window misses the frame."""
    from monkey_pose_b200 import tf_monkeydetector as tmd
    rng = np.random.default_rng(11)
    n, h, w = 300, 424, 512
    base = np.round(rng.uniform(600, 4000, size=(4, h, w)) / 8) * 8
    frames = torch.as_tensor((base[rng.integers(0, 4, n)] / 10000.0).astype(np.float32)).cuda()
    tr = np.stack([rng.uniform(-0.2, 1.4, n), rng.uniform(-0.2, 1.2, n), rng.uniform(0.03, 0.5, n)], 1).astype(np.float32)
    tr[7] = [np.nan, 0.5, 0.2]
    tr[8] = [0.5, 0.5, 0.0]
    md_h = tmd.tfMonkeyDetector(365.456, 365.456, 256, 212, [800, 800, 1200], 200, 10000)
    md_d = tmd.tfMonkeyDetector(365.456, 365.456, 256, 212, [800, 800, 1200], 200, 10000)
    with np.errstate(all="ignore"):
        p_h, c_h, M_h = tmd.prepare_data_test(frames, tr, md_h, _Cfg())
    p_d, c_d, M_d = tmd.prepare_data_test(frames, torch.as_tensor(tr).cuda(), md_d, _Cfg())
    bad_h = np.zeros(n, bool)
    bad_h[md_h.last_invalid] = True
    bad_d = md_d.last_invalid_dev.cpu().numpy().astype(bool)
    assert np.array_equal(bad_h, bad_d) and 10 < bad_h.sum() < n - 10
    assert torch.equal(p_h, p_d)
    good = ~bad_h
    assert np.array_equal(np.asarray(c_h)[good], c_d.cpu().numpy()[good])
    assert np.array_equal(np.asarray(M_h)[good], M_d.cpu().numpy()[good])
    ip_d, zp_d = md_d._last_windows_dev
    ints, z, _ = md_h._windows_batch(np.asarray(c_h), h, w, (128, 128))
    assert np.array_equal(ip_d.cpu().numpy()[good], ints[good]) and np.array_equal(zp_d.cpu().numpy()[good], z[good])
    # the device centres feed the post-processing directly
    out = torch.rand(n, 69, device="cuda") - 0.5
    xyz_h, uvd_h = md_h.getAbsoluteCoordinates_batch(out, c_h, 600.0)
    xyz_d, uvd_d = md_d.getAbsoluteCoordinates_batch(out, c_d, 600.0)
    assert torch.equal(xyz_h[good], xyz_d[good]) and torch.equal(uvd_h[good], uvd_d[good])


def test_frames_to_joints_pipeline_equals_the_stage_by_stage_sequence():
    """FramesToJoints (chunked upload on a copy stream, attention CNN per chunk, device-side window arithmetic, pose
    network, absolute coordinates) against the same stages called one after the other on resident frames: bitwise."""
    from monkey_pose_b200 import tf_monkeydetector as tmd
    rng = np.random.default_rng(21)
    n, h, w = 16, 424, 512
    base = np.round(rng.uniform(600, 4000, size=(4, h, w)) / 8) * 8
    frames_np = (base[rng.integers(0, 4, n)] / 10000.0).astype(np.float32)
    centres = np.stack([rng.uniform(0.3, 0.9, n), rng.uniform(0.25, 0.7, n), rng.uniform(0.1, 0.3, n)], 1).astype(np.float32)
    md = tmd.tfMonkeyDetector(365.456, 365.456, 256, 212, [800, 800, 1200], 200, 10000)
    am = mp.attn_model_struct()
    am.widths, am.fc_hidden = (8, 8, 8, 8, 8), 16
    am.load_params(init.attn_params(widths=am.widths, fc_hidden=16, out=3, seed=8))
    pm = mp.model()
    pm.channels, pm.timesteps, pm.fc_hidden = 25, 2, 32
    pm.hidden_state = init.hidden_init((n, 64, 64, 25), seed=5)
    pm.load_params(init.pose_params(channels=25, S=15, T=2, hw=64, fc_hidden=32, out=69, seed=3, stress=4.0))
    c_dev = torch.as_tensor(centres).cuda()
    pipe = mp.FramesToJoints(am, pm, md, _Cfg(), cube_z=1200.0, chunks=4)
    xyz, uvd = pipe(torch.as_tensor(frames_np).pin_memory(), centres=c_dev)
    xyz2, uvd2 = pipe(torch.as_tensor(frames_np).pin_memory(), centres=c_dev)          # buffers are reused
    assert torch.equal(xyz, xyz2) and torch.equal(uvd, uvd2)
    # the attention CNN ran on every chunk (its split-K layout follows the batch size, so chunks of 4 frames and one
    # batch of 16 agree to rounding, not bit for bit)
    f_dev = torch.as_tensor(frames_np).cuda()
    tr_ref = am.build(f_dev, 3)
    assert torch.allclose(pipe._tr, tr_ref, rtol=1e-4, atol=1e-6)
    p, cs, _ = tmd.prepare_data_test(f_dev, c_dev, md, _Cfg())
    x_ref, u_ref = md.getAbsoluteCoordinates_batch(pm.build(p, 69), cs, 600.0)
    assert torch.equal(xyz, x_ref.cpu()) and torch.equal(uvd, u_ref.cpu())
    assert xyz.shape == (n, 23, 3) and torch.isfinite(xyz).all()
    # driven by the attention output itself (random-init: most windows miss the frame -> background patches, still finite)
    xyz3, _ = pipe(torch.as_tensor(frames_np).pin_memory())
    assert torch.isfinite(xyz3).all()
    # raw 16-bit millimetre frames (the real-data loop, train_cnn_networks_hgru.py:381-386): thresholds and the division
    # run on the device; same result as the host pre-processing followed by the float32 path, bit for bit
    raw = np.round(frames_np * 10000.0).astype(np.uint16)
    im = raw.astype(np.float64)
    im[im < 1000] = 10000
    im[im > 3000] = 10000
    host_frames = (im / 10000.0).astype(np.float32)
    dev = tmd.preprocess_real_depth(torch.from_numpy(raw.view(np.int16)).cuda())
    assert np.array_equal(dev.cpu().numpy(), host_frames)
    xa, ua = pipe(torch.from_numpy(raw.view(np.int16)).pin_memory(), centres=c_dev)
    xb, ub = pipe(torch.as_tensor(host_frames).pin_memory(), centres=c_dev)
    assert torch.equal(xa, xb) and torch.equal(ua, ub)


# ---- post-processing (SURVEY 8f rank 2) -------------------------------------------------------------
def test_postprocess_bit_exact_against_reference_golden():
    from monkey_pose_b200 import pose_evaluation as pe
    from monkey_pose_b200 import tf_monkeydetector as tmd
    z = np.load(os.path.join(GOLDEN, "post_ref.npz"))
    md = tmd.tfMonkeyDetector(365.456, 365.456, 256, 212, [800, 800, 1200], 200, 10000)
    xyz, uvd = md.getAbsoluteCoordinates_batch(torch.as_tensor(z["out_put"]).cuda(), z["coms"], float(z["scale"]))
    assert np.array_equal(xyz.cpu().numpy(), z["xyz"])
    assert np.array_equal(uvd.cpu().numpy(), z["uvd"])
    n = z["out_put"].shape[0]
    res = torch.as_tensor(np.reshape(z["out_put"], (n, -1, 3)) * np.float32(z["scale"])).cuda()
    lab = torch.as_tensor(np.reshape(z["labels"], (n, -1, 3)) * np.float32(z["scale"])).cuda()
    assert abs(pe.getMeanError_np(lab, res) - float(z["mean_error_mm"])) <= 1e-5 * float(z["mean_error_mm"])
    assert pe.getMaxError_np(lab, res) == float(z["max_error_mm"])
    lab[0, 0, 0] = float("nan")                       # NaN joints are skipped like numpy.nanmean
    assert np.isfinite(pe.getMeanError_np(lab, res))
    # single-frame host methods mirror the reference API too
    a, b = md.getAbsoluteCoordinates(z["xyz"][0] - md.uvdtoxyz(z["coms"][0]), z["coms"][0])
    assert np.allclose(b, z["uvd"][0], rtol=1e-5, atol=1e-3)


# ---- attention (centre-of-mass) CNN (SURVEY 8f rank 4) ----------------------------------------------
def _attn_golden():
    z = np.load(os.path.join(GOLDEN, "attn_ref.npz"))
    return z["frames"], {k[4:]: z[k] for k in z.files if k.startswith("var:")}, \
        {k[4:]: z[k] for k in z.files if k.startswith("act:")}


@pytest.mark.gpu
def test_attn_model_matches_reference_golden_every_layer():
    """attn_model_struct against the outputs of the reference's own class (tests/golden/make_golden_attn.py):
    the resize bit for bit, every pooled feature map and the head within the split-bf16 budget."""
    frames, P, A = _attn_golden()
    m = mp.attn_model_struct()
    m.load_params(P)
    out = m.build(torch.as_tensor(frames).cuda(), 3, train_mode=False)
    assert out.shape == (2, 3) and m.gpu_launches > 0
    assert np.array_equal(m.activation("resized").cpu().numpy()[..., 0], A["resized"][..., 0])
    for k in ("pool1", "pool2", "pool3", "pool4", "pool5"):
        assert onp.rel_err(getattr(m, k).cpu().numpy(), A[k])[0] < 1e-4, k
    assert onp.rel_err(m.fc1.cpu().numpy(), A["fc1"])[0] < 1e-4
    assert onp.rel_err(out.cpu().numpy(), A["out_put"])[0] < 1e-4


@pytest.mark.gpu
@pytest.mark.parametrize("cfg", [(3, 424, 512, (64, 128, 256, 512, 1024), 1024), (5, 96, 80, (8, 24, 16, 40, 32), 64)])
def test_attn_model_vs_oracle(cfg):
    """Reference widths on Kinect-size frames (and an odd small configuration) against the fp64 torch oracle."""
    from oracle import attn_oracle_torch as atorch
    N, H, W, widths, F = cfg
    P = init.attn_params(widths, F, 3, seed=5, random_bn=True)
    rng = np.random.default_rng(3)
    frames = rng.uniform(0.06, 0.4, size=(N, H, W, 1)).astype(np.float32)
    frames[rng.uniform(size=frames.shape) < 0.05] = 0.0
    m = mp.attn_model_struct()
    m.load_params(P)
    out = m.build(torch.as_tensor(frames).cuda(), 3)
    ref, acts = atorch.attn_forward(frames, P, dtype=torch.float64, trace=True)
    assert onp.rel_err(m.pool3.cpu().numpy(), acts["pool3"].numpy())[0] < 1e-4
    assert onp.rel_err(m.pool5.cpu().numpy(), acts["pool5"].numpy())[0] < 1e-4
    assert onp.rel_err(out.cpu().numpy(), ref.numpy())[0] < 1e-4
    # determinism + the error convention of the mirror
    assert torch.equal(out, m.build(torch.as_tensor(frames).cuda(), 3))
    with pytest.raises(RuntimeError):
        m.build(torch.as_tensor(frames), 3)


# ---- bf16x3: fp32-class accuracy on tensor cores (hi/lo operand splits), k <= 32, S = 15 -------------------
@pytest.mark.gpu
def test_bf16x3_mode_matches_reference_golden_every_timestep():
    z = np.load(os.path.join(GOLDEN, "hgru_ref_S15_k8.npz"))
    T, S = int(z["T"]), int(z["S"])
    params = {n: z["var:contextual_circuit/" + n] for n in onp.HGRU_PARAM_NAMES}
    cc, O, _ = _run_cc(z["X"], z["O0"], params, T, S, "bf16x3")
    for t in range(T):
        assert onp.rel_err(cc.I_steps[t].cpu().numpy(), z["I_steps"][:, t])[0] < 1e-4, t
        assert onp.rel_err(cc.O_steps[t].cpu().numpy(), z["O_steps"][:, t])[0] < 1e-4, t
    assert onp.rel_err(O.cpu().numpy(), z["O_final"])[0] < 1e-4


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(2, 64, 64, 25, 15, 2), (1, 20, 36, 32, 15, 3), (1, 33, 70, 16, 15, 2),
                                   (1, 64, 64, 64, 15, 2), (2, 19, 21, 48, 15, 2), (1, 37, 45, 64, 15, 2)])
def test_bf16x3_mode_seeded_cases_vs_oracle(shape):
    """Stress weights (tanh off its linear region): the split-bf16 tensor-core path stays inside the fp32 budget
    that plain bf16 misses by two orders of magnitude."""
    n, h, w, k, S, T = shape
    rng = np.random.default_rng(5)
    X = rng.uniform(-1, 1, size=(n, h, w, k)).astype(np.float32)
    O0 = init.hidden_init((n, h, w, k), seed=3, limit=0.5)
    params = init.hgru_params(k, S, T, seed=9, stress=6.0)
    cc, O, _ = _run_cc(X, O0, params, T, S, "bf16x3")
    ref, H1s, H2s = otorch.hgru_forward(X, O0, params, T, dtype=torch.float64, trace=True)
    for t in range(T):
        assert onp.rel_err(cc.I_steps[t].cpu().numpy(), H1s[t].numpy())[0] < 1e-4
        assert onp.rel_err(cc.O_steps[t].cpu().numpy(), H2s[t].numpy())[0] < 1e-4
    assert onp.rel_err(O.cpu().numpy(), ref.numpy())[0] < 1e-4


@pytest.mark.gpu
def test_bf16x3_pose_model_and_unsupported_shapes():
    m, out, P, depth, h0 = _pose("bf16x3", 2, 25, 16, 2, 15, 64)
    ref = otorch.pose_forward(depth, P, h0, timesteps=2, dtype=torch.float64)
    assert onp.rel_err(out.cpu().numpy(), ref.numpy())[0] < 1e-4
    assert onp.mean_joint_error_mm(out.cpu().numpy(), ref.numpy()) < 0.01
    with pytest.raises(NotImplementedError):          # only the 15x15 horizontal kernel is instantiated
        _pose("bf16x3", 1, 16, 16, 1, 5, 32)


@pytest.mark.parametrize("mode", ["bf16", "fp32"])
def test_streamed_forward_equals_batch_by_batch_build(mode):
    """StreamedForward (upload of batch i+1 and read-back of batch i-1 around the forward of batch i) yields, in
    order, bitwise what model.build returns for each host batch; buffers are reused safely over more than two
    batches, and a second pass over the same object restarts cleanly."""
    N, ch, hw, T, S, F = 5, 16, 16, 2, 15, 32
    m, _, P, _, _ = _pose(mode, N, ch, hw, T, S, F)
    m.hidden_state, m.aux = None, dict(m.aux, hidden_init="zeros")      # (any batch size: the ragged case below)
    batches = [torch.as_tensor(init.synthetic_depth(N, seed=10 + i, size=2 * hw)).pin_memory() for i in range(5)]
    want = [m.build(b, 69).clone() for b in batches]
    assert not torch.equal(want[0], want[1])
    sf = mp.StreamedForward(m, 69)
    for _ in range(2):
        got = list(sf(iter(batches)))
        assert len(got) == len(want)
        for g, w in zip(got, want):
            assert not g.is_cuda and torch.equal(g, w)
    assert list(sf(iter([]))) == []
    with pytest.raises(ValueError):
        list(sf([batches[0].cuda()]))
    # a ragged last batch (new shape mid-stream): what is in flight is handed out first, then new buffers
    ragged = batches[:3] + [batches[3][:2]]
    got = list(sf(iter(ragged)))
    assert [tuple(g.shape) for g in got] == [(N, 69)] * 3 + [(2, 69)]
    for g, w in zip(got[:3], want[:3]):
        assert torch.equal(g, w)
    assert torch.equal(got[3], m.build(batches[3][:2].contiguous().pin_memory(), 69))


@pytest.mark.gpu
@pytest.mark.parametrize("path", HGRU_FILES, ids=[os.path.basename(p) for p in HGRU_FILES])
def test_stepping_the_circuit_by_hand_matches_reference_golden(path):
    """The reference's per-timestep methods (circuit_input, input_integration, circuit_output, output_integration,
    full, condition; hgru_module.py:692-861) as stand-alone exact-fp32 ops: driving `full()` in a Python loop
    reproduces the reference-produced H1 / H2 of every timestep, and the fused `build()` of the same circuit."""
    z = np.load(path)
    T, S = int(z["T"]), int(z["S"])
    if z["X"].shape[3] > 32 and z["X"].shape[1] * z["X"].shape[2] > 1024:
        pytest.skip("direct 15x15 convolution at 64 channels: covered by the smaller fixtures")
    params = {n: z["var:contextual_circuit/" + n] for n in onp.HGRU_PARAM_NAMES}
    cc = mp.ContextualCircuit(X=torch.as_tensor(z["X"]).cuda(), timesteps=T, SRF=1, SSN=S, SSF=S, aux=POSE_AUX,
                              params=params, hidden_state=z["O0"], compute_mode="fp32")
    cc.prepare_tensors()
    O = torch.as_tensor(z["O0"]).cuda()
    I = torch.zeros_like(O)
    i0, store_I, store_O = 0, None, None
    while cc.condition(i0, O, I, store_I, store_O):
        O_before = O.clone()
        t = i0
        i0, O, I, store_I, store_O = cc.full(i0, O, I, store_O, store_I)
        assert onp.rel_err(I.cpu().numpy(), z["I_steps"][:, t])[0] < 1e-5, t
        assert onp.rel_err(O.cpu().numpy(), z["O_steps"][:, t])[0] < 1e-5, t
        assert torch.equal(O_before, O_before.clone()) and O.data_ptr() != O_before.data_ptr()
    assert i0 == T
    assert onp.rel_err(O.cpu().numpy(), z["O_final"])[0] < 1e-5
    fused, _, _ = cc.build()
    assert onp.rel_err(O.cpu().numpy(), fused.cpu().numpy())[0] < 1e-5
    # the pieces on their own: the gate leaves its input alone, conv_2d_op is the plain cross-correlation
    O0 = torch.as_tensor(z["O0"]).cuda()
    keep = O0.clone()
    P, G1 = cc.circuit_input(O0)
    assert torch.equal(O0, keep)
    ref_P = onp.conv2d_same(z["O0"].astype(np.float64) * G1.cpu().numpy().astype(np.float64),
                            params["p_r"].astype(np.float64)) + params["lateral_bias"].astype(np.float64)
    assert onp.rel_err(P.cpu().numpy(), ref_P)[0] < 1e-5
    plain = cc.conv_2d_op(data=O0, weight_key="p_r")
    assert onp.rel_err((plain + cc.lateral_bias).cpu().numpy(), cc.process_p(O0, "p_r", None).cpu().numpy())[0] < 1e-6
    cc.conv_2d_op(data=O0, weight_key="i_r", out_key="I_r")
    assert tuple(cc.I_r.shape) == tuple(O0.shape)
