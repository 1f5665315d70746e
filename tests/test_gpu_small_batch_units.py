"""Small batches run the hGRU's 15x15 conv launches on narrow units (1 output tile instead of 8 on the tap-stacked
kernel, 2 tiles instead of 4 on the fused 64-channel kernel) so that a few frames occupy more SMs.  The width is
picked from the batch size alone and must not change any value: a frame's result is bitwise the same whether it runs
alone on narrow units or inside a batch large enough for wide ones."""
import ctypes

import numpy as np
import pytest
import torch

import monkey_pose_b200 as mp
from monkey_pose_b200 import _lib
from monkey_pose_b200 import initialization as init

HW, S, F, O = 64, 15, 64, 69
BIG = 256
ISSUE_NS = (1, 2, 3, 5, 8, 16, 18, 19, 20, 36, 37, 38)


def _st():
    return torch.cuda.current_stream().cuda_stream


def _ptr(t):
    return None if t is None else t.data_ptr()


def _cdiv(a, b):
    return -(-a // b)


def _narrow(n, H, W, ch, sms):
    """Mirror of the library's unit-width rule (narrow_units_faster in lib_common.cuh and its callers): narrow when
    waves x tensor-core instructions per unit is strictly smaller than with wide units."""
    uy = _cdiv(H, 16)
    if ch <= 32:      # tap-stacked kernel: work = tiles per unit, the carry tile included
        wide, narrow = n * _cdiv(W, 64) * uy, n * _cdiv(W, 8) * uy
        return _cdiv(narrow, sms) * 2 < _cdiv(wide, sms) * (1 + _cdiv(min(W, 64), 8))
    wide, narrow = n * _cdiv(W, 32) * uy, n * _cdiv(W, 16) * uy      # fused paired-tap kernel: 8 UT + 7 per row
    return _cdiv(narrow, sms) * 23 < _cdiv(wide, sms) * 39


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _batch_sizes(ch):
    """The issue's sizes plus the last narrow and the first wide batch on this device."""
    sms = _sms()
    last = max(n for n in range(1, BIG + 1) if _narrow(n, HW, HW, ch, sms))
    ns = sorted(set(ISSUE_NS) | {last, last + 1})
    assert any(_narrow(n, HW, HW, ch, sms) for n in ns) and not all(_narrow(n, HW, HW, ch, sms) for n in ns)
    assert not _narrow(BIG, HW, HW, ch, sms)
    return ns


def _pose_plan(mode, ch, T_, depth):
    m = mp.model()
    m.channels, m.timesteps, m.SSF, m.SSN, m.fc_hidden, m.compute_mode = ch, T_, S, S, F, mode
    m.aux = dict(m.aux, hidden_init="zeros")
    m.load_params(init.pose_params(channels=ch, S=S, T=T_, hw=HW, fc_hidden=F, out=O, seed=3, stress=4.0,
                                   random_bn=True))
    m.build(depth, O)
    torch.cuda.synchronize()
    return m


def _pose_run(plan, n, depth, h0, ch):
    lib = _lib.load()
    out = torch.full((n, O), float("nan"), device="cuda")
    _lib.check(lib.pose_forward_batch(plan, n, depth.data_ptr(), _ptr(h0), out.data_ptr(), _st()),
               "pose_forward_batch")
    acts = {}
    for name, per in (("hgru", HW * HW * ch), ("fc1", F)):
        dst = torch.full((n * per,), float("nan"), device="cuda")
        _lib.check(lib.pose_get_activation(plan, name.encode(), dst.data_ptr(), _st()), "pose_get_activation")
        acts[name] = dst.view(n, per)
    torch.cuda.synchronize()
    return out, acts, lib.pose_plan_launch_count(plan)


POSE_CASES = [(mode, ch, T_) for mode in ("bf16", "fp16") for ch, T_ in ((25, 2), (32, 16), (64, 2))] + \
             [("bf16x3", 25, 2), ("bf16x3", 32, 16)]


@pytest.mark.gpu
@pytest.mark.parametrize("mode,ch,T_", POSE_CASES)
def test_small_batches_equal_their_frames_of_a_full_batch(mode, ch, T_):
    """pose_forward_batch at each n equals frames [off, off + n) of one n = 256 forward on the same plan: the
    predictions and the hgru / fc1 activations, bit for bit; launch counts equal."""
    depth = torch.as_tensor(init.synthetic_depth(BIG, seed=11, size=2 * HW)).cuda()
    h0 = torch.as_tensor(init.hidden_init((BIG, HW, HW, ch), seed=5, limit=0.3)).cuda()
    m = _pose_plan(mode, ch, T_, depth)
    full_out, full_acts, full_launches = _pose_run(m._plan, BIG, depth, h0, ch)
    assert torch.isfinite(full_out).all()
    for n in _batch_sizes(ch):
        off = (37 * n + 11) % (BIG - n + 1)
        out, acts, launches = _pose_run(m._plan, n, depth[off:off + n].contiguous(), h0[off:off + n].contiguous(), ch)
        assert torch.equal(out, full_out[off:off + n]), (n, off)
        for name in acts:
            assert torch.equal(acts[name], full_acts[name][off:off + n]), (n, off, name)
        assert launches == full_launches, n


@pytest.mark.gpu
@pytest.mark.parametrize("ch", [25, 64])
def test_launch_count_does_not_depend_on_the_unit_width(ch):
    depth = torch.as_tensor(init.synthetic_depth(BIG, seed=2, size=2 * HW)).cuda()
    m = _pose_plan("bf16", ch, 3, depth)
    counts = [_pose_run(m._plan, n, depth[:n].contiguous(), None, ch)[2] for n in (1, BIG)]
    assert counts[0] == counts[1] > 0


def _hgru_plan(n, H, W, k, T_, mode, params):
    lib = _lib.load()
    h = ctypes.c_void_p()
    _lib.check(lib.hgru_plan_create(n, H, W, k, S, T_, _lib.MODES[mode], ctypes.byref(h)), "hgru_plan_create")
    ptrs = [params[name].data_ptr() for name in _lib.HGRU_PARAM_ORDER]
    _lib.check(lib.hgru_set_params(h, *ptrs, _st()), "hgru_set_params")
    return h


def _hgru_run(plan, n, X, O0, trace, T_):
    lib = _lib.load()
    out = torch.full((n,) + tuple(X.shape[1:]), float("nan"), device="cuda")
    tr = [torch.full((T_, n) + tuple(X.shape[1:]), float("nan"), device="cuda") for _ in range(2)] if trace \
        else [None, None]
    _lib.check(lib.hgru_forward_batch(plan, n, X.data_ptr(), _ptr(O0), out.data_ptr(), _ptr(tr[0]), _ptr(tr[1]),
                                      _st()), "hgru_forward_batch")
    torch.cuda.synchronize()
    return out, tr


@pytest.mark.gpu
@pytest.mark.parametrize("mode,k", [("bf16", 25), ("bf16", 32), ("bf16", 64), ("fp16", 25), ("fp16", 32),
                                    ("fp16", 64), ("bf16x3", 25), ("bf16x3", 32)])
def test_hgru_single_frame_equals_its_frame_of_a_wide_unit_forward(mode, k):
    """A ContextualCircuit-sized plan with W = 60, a multiple of neither unit width: one frame (narrow units) equals
    the same frame inside a 148-frame forward (wide units), chained, and at every timestep of the H1 / H2 traces."""
    H, W, T_, cap, off = 30, 60, 3, 148, 77
    sms = _sms()
    assert _narrow(1, H, W, k, sms) and not _narrow(cap, H, W, k, sms)
    rng = np.random.default_rng(21)
    X = torch.as_tensor(rng.uniform(-1, 1, size=(cap, H, W, k)).astype(np.float32)).cuda()
    O0 = torch.as_tensor(init.hidden_init((cap, H, W, k), seed=4, limit=0.5)).cuda()
    params = {n: torch.as_tensor(np.asarray(v, np.float32)).cuda()
              for n, v in init.hgru_params(k, S, T_, seed=9, stress=6.0).items()}
    plan = _hgru_plan(cap, H, W, k, T_, mode, params)
    try:
        for trace in (False, True):      # untraced forwards are chained, traced ones stream-ordered
            full = _hgru_run(plan, cap, X, O0, trace, T_)
            one = _hgru_run(plan, 1, X[off:off + 1].contiguous(), O0[off:off + 1].contiguous(), trace, T_)
            assert torch.isfinite(full[0]).all()
            assert torch.equal(one[0], full[0][off:off + 1]), trace
            if trace:
                for a, b in zip(one[1], full[1]):
                    for t in range(T_):
                        assert torch.equal(a[t], b[t, off:off + 1]), t
    finally:
        _lib.load().hgru_plan_destroy(plan)
