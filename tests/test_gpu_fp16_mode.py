"""compute_mode='fp16': the bf16 tensor-core pipeline with IEEE fp16 conv operands (11 significand bits instead of 8).

GPU (B200): per timestep against the fp64 oracle at the baseline configs, at a quarter of the tensor-core budget and
at most half the bf16 mode's error on the same inputs; the reference-source goldens; the whole pose forward at batch
256 (host entry, sub-batches); an initial state beyond fp16 range.  CPU: the mode's constant and its shape checks,
which run before any CUDA call."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

import monkey_pose_b200 as mp
from monkey_pose_b200 import initialization as init
from oracle import hgru_oracle_np as onp
from oracle import hgru_oracle_torch as otorch
from tests.test_gpu_parity_baseline import GOLDEN, LAYER_CASES, POSE_AUX, SUBSET, WEIGHT_SETS, _layer_case, _model, \
    _pose_case

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TOL = 2.5e-3        # a quarter of the 1e-2 budget of the bf16 tensor-core path
MM_TOL = 0.1        # mean per-joint deviation, mm


# ---- CPU ------------------------------------------------------------------------------------------------------------
def test_fp16_mode_constant_matches_header():
    src = open(os.path.join(ROOT, "include", "hgru_b200.h")).read()
    m = re.search(r"#define\s+HGRU_MODE_FP16\s+(\d+)", src)
    assert m, "HGRU_MODE_FP16 not defined"
    assert mp._lib.MODES["fp16"] == mp._lib.MODE_FP16 == int(m.group(1))


def test_fp16_plan_rejects_unsupported_shapes_before_cuda():
    """S != 15 and k > 64: HGRU_E_UNSUPPORTED (NotImplementedError in Python) from argument checks that need no
    device."""
    lib = mp._lib.load()
    fp16 = mp._lib.MODE_FP16
    h = ctypes.c_void_p()
    assert lib.hgru_plan_create(1, 8, 8, 8, 5, 1, fp16, ctypes.byref(h)) == 2
    assert b"fp16" in lib.hgru_last_error()
    assert lib.hgru_plan_create(1, 8, 8, 65, 15, 1, fp16, ctypes.byref(h)) == 2
    with pytest.raises(NotImplementedError):
        mp._lib.check(lib.hgru_plan_create(1, 8, 8, 8, 7, 1, fp16, ctypes.byref(h)), "hgru_plan_create")


# ---- GPU: the recurrent layer -----------------------------------------------------------------------------------------
def _traced(X, O0, params, T, mode):
    cc = mp.ContextualCircuit(X=torch.as_tensor(X).cuda(), timesteps=T, SRF=1, SSN=15, SSF=15, aux=POSE_AUX,
                              params=params, hidden_state=O0, compute_mode=mode)
    O, _, _ = cc.build(trace=True)
    torch.cuda.synchronize()
    return O, [h.cpu().numpy() for h in cc.I_steps], [h.cpu().numpy() for h in cc.O_steps]


@pytest.mark.gpu
@pytest.mark.parametrize("wset", sorted(WEIGHT_SETS))
@pytest.mark.parametrize("case", sorted(LAYER_CASES))
def test_fp16_every_timestep_vs_fp64_oracle(case, wset):
    k, T = LAYER_CASES[case]
    X, O0, params, ref, H1s, H2s = _layer_case(case, wset)
    O, I_steps, O_steps = _traced(X, O0, params, T, "fp16")
    for t in range(T):
        e1, e2 = onp.rel_err(I_steps[t], H1s[t])[0], onp.rel_err(O_steps[t], H2s[t])[0]
        assert e1 <= TOL and e2 <= TOL, (case, wset, t, e1, e2)
    assert onp.rel_err(O.cpu().numpy(), ref)[0] <= TOL
    # the untraced forward (chained launches) gives the same final state, bit for bit
    O2, _, _ = mp.ContextualCircuit(X=torch.as_tensor(X).cuda(), timesteps=T, SRF=1, SSN=15, SSF=15, aux=POSE_AUX,
                                    params=params, hidden_state=O0, compute_mode="fp16").build()
    assert torch.equal(O2, O)


def _worst(case, wset, mode):
    k, T = LAYER_CASES[case]
    X, O0, params, ref, H1s, H2s = _layer_case(case, wset)
    O, I_steps, O_steps = _traced(X, O0, params, T, mode)
    errs = [max(onp.rel_err(I_steps[t], H1s[t])[0], onp.rel_err(O_steps[t], H2s[t])[0]) for t in range(T)]
    return max(errs + [onp.rel_err(O.cpu().numpy(), ref)[0]])


# Where fp16 operands do not halve the bf16 mode's worst error (measured on a B200, DESIGN.md section 4 "fp32 vs tf32
# vs fp16"): the errors of both modes there are close to each other, i.e. set by something the two modes share.
_NOT_HALVED = {("k32_T16", "random_init"): "fp16 / bf16 = 0.95", ("k32_T16", "stress"): "fp16 / bf16 = 0.80",
               ("k64_T8", "random_init"): "fp16 / bf16 = 0.52"}


@pytest.mark.gpu
@pytest.mark.parametrize("case,wset", [
    pytest.param(c, w, marks=pytest.mark.xfail(strict=True, reason=_NOT_HALVED[(c, w)])) if (c, w) in _NOT_HALVED
    else (c, w) for c in sorted(LAYER_CASES) for w in sorted(WEIGHT_SETS)])
def test_fp16_at_most_half_the_bf16_error(case, wset):
    worst = {mode: _worst(case, wset, mode) for mode in ("bf16", "fp16")}
    print("%s %s: worst per-timestep rel err fp16 %.3e, bf16 %.3e (ratio %.2f)"
          % (case, wset, worst["fp16"], worst["bf16"], worst["fp16"] / worst["bf16"]))
    assert worst["fp16"] < worst["bf16"]
    assert worst["fp16"] <= 0.5 * worst["bf16"], worst


@pytest.mark.gpu
@pytest.mark.parametrize("tag", ["S15_k25_T8", "S15_k25_T8_stress", "S15_k32_T16_stress", "S15_k64_T3_stress"])
def test_fp16_reference_source_goldens(tag):
    z = np.load(os.path.join(GOLDEN, "hgru_ref_%s.npz" % tag))
    T, S = int(z["T"]), int(z["S"])
    params = {n: z["var:contextual_circuit/" + n] for n in onp.HGRU_PARAM_NAMES}
    O, I_steps, O_steps = _traced(z["X"], z["O0"], params, T, "fp16")
    for t in range(T):
        e1 = onp.rel_err(I_steps[t], z["I_steps"][:, t])[0]
        e2 = onp.rel_err(O_steps[t], z["O_steps"][:, t])[0]
        assert e1 <= TOL and e2 <= TOL, (tag, t, e1, e2)
    assert onp.rel_err(O.cpu().numpy(), z["O_final"])[0] <= TOL


@pytest.mark.gpu
def test_fp16_initial_state_beyond_fp16_range_stays_finite():
    """A unit-range initial state x 1e5 (beyond +-65504): the first gated operand saturates instead of turning into
    inf, so every H1 and H2 stays finite."""
    X, O0, params, _, _, _ = _layer_case("k25_T8", "stress")
    O0 = O0 / np.abs(O0).max() * 1e5
    assert np.abs(O0).max() > 65504
    O, I_steps, O_steps = _traced(X, O0, params, 8, "fp16")
    for t in range(8):
        assert np.isfinite(I_steps[t]).all() and np.isfinite(O_steps[t]).all(), t
    assert torch.isfinite(O).all()


# ---- GPU: the whole pose model ----------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("stress,random_bn", [(1.0, False), (4.0, True)], ids=["random_init", "stress"])
def test_fp16_pose_forward_batch256_vs_fp64_oracle(stress, random_bn):
    P, depth, h0, ref, acts = _pose_case(stress, random_bn)
    idx = list(SUBSET)
    m = _model(P, h0, 25, 8, "fp16")
    out = m.build(torch.as_tensor(depth).cuda(), 69)
    torch.cuda.synchronize()
    got = out.cpu().numpy()
    assert np.isfinite(got).all()
    e = onp.rel_err(got[idx], ref)[0]
    mm = onp.mean_joint_error_mm(got[idx], ref)
    eh = onp.rel_err(m.activation("hgru").cpu().numpy()[idx], acts["hgru"])[0]
    print("pose N=256 fp16 (stress %g): out_put rel %.3e, %.4f mm, hgru rel %.3e" % (stress, e, mm, eh))
    assert e <= TOL and eh <= TOL and mm <= MM_TOL
    out_host = m.build(torch.as_tensor(depth).pin_memory(), 69)
    assert not out_host.is_cuda and np.array_equal(out_host.numpy(), got)
    sub = _model(P, h0[idx], 25, 8, "fp16").build(torch.as_tensor(depth[idx]).cuda(), 69)
    assert np.array_equal(sub.cpu().numpy(), got[idx])


@pytest.mark.gpu
def test_fp16_pose_forward_reference_width_and_deep_variant_vs_fp64_oracle():
    for ch, T in ((64, 8), (32, 16)):
        N, hw, F = 8, 64, 256
        P = init.pose_params(channels=ch, S=15, T=T, hw=hw, fc_hidden=F, out=69, seed=3, stress=4.0, random_bn=True)
        depth = init.synthetic_depth(N, seed=77, size=128)
        h0 = init.hidden_init((N, hw, hw, ch), seed=5)
        idx = [0, 7]
        ref = otorch.pose_forward(depth[idx], P, h0[idx], timesteps=T, dtype=torch.float64).numpy()
        m = _model(P, h0, ch, T, "fp16")
        m.fc_hidden = F
        got = m.build(torch.as_tensor(depth).cuda(), 69).cpu().numpy()
        e, mm = onp.rel_err(got[idx], ref)[0], onp.mean_joint_error_mm(got[idx], ref)
        print("pose k=%d T=%d fp16: out_put rel %.3e, %.4f mm" % (ch, T, e, mm))
        assert e <= TOL and mm <= MM_TOL
