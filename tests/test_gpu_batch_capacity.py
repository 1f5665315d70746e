"""Batches of any size up to a plan's capacity: pose_forward_batch, pose_forward_host_batch, hgru_forward_batch and
attn_forward_batch run the first n frames of a plan created for N >= n frames.  The result must equal that of a
plan created for exactly n frames, bit for bit, and the Python mirrors must keep one plan while the batch size
changes below its capacity."""
import ctypes

import numpy as np
import pytest
import torch

import monkey_pose_b200 as mp
from monkey_pose_b200 import _lib
from monkey_pose_b200 import hgru_module as hm
from monkey_pose_b200 import initialization as init

HW, T, S, F, O = 64, 2, 15, 64, 69
ACT_NAMES = ("pool1", "conv2", "conv3", "hgru", "fc1")


def _st():
    return torch.cuda.current_stream().cuda_stream


def _ptr(t):
    return None if t is None else t.data_ptr()


def _pose_model(mode, ch, depth, seed=3):
    """A model whose plan was created (and its parameters set) for depth.shape[0] frames."""
    m = mp.model()
    m.channels, m.timesteps, m.SSF, m.SSN, m.fc_hidden, m.compute_mode = ch, T, S, S, F, mode
    m.aux = dict(m.aux, hidden_init="zeros")
    m.load_params(init.pose_params(channels=ch, S=S, T=T, hw=HW, fc_hidden=F, out=O, seed=seed, stress=4.0,
                                   random_bn=True))
    m.build(depth, O)
    torch.cuda.synchronize()
    return m


def _pose_run(plan, n, depth, h0, identity, ch, batch=True):
    """One forward of n frames on `plan`: output, launch count and every activation (with 16 NaN guard values
    behind the n frames)."""
    lib = _lib.load()
    _lib.check(lib.pose_set_hidden_init(plan, 1 if identity else 0), "pose_set_hidden_init")
    out = torch.full((n, O), float("nan"), device="cuda")
    if batch:
        _lib.check(lib.pose_forward_batch(plan, n, depth.data_ptr(), _ptr(h0), out.data_ptr(), _st()),
                   "pose_forward_batch")
    else:
        _lib.check(lib.pose_forward(plan, depth.data_ptr(), _ptr(h0), out.data_ptr(), _st()), "pose_forward")
    launches = lib.pose_plan_launch_count(plan)
    acts = {}
    for name in ACT_NAMES:
        numel = n * F if name == "fc1" else n * HW * HW * ch
        dst = torch.full((numel + 16,), float("nan"), device="cuda")
        _lib.check(lib.pose_get_activation(plan, name.encode(), dst.data_ptr(), _st()), "pose_get_activation")
        acts[name] = dst
    torch.cuda.synchronize()
    return out, launches, acts


def _same_acts(a, b, n, ch):
    for name in ACT_NAMES:
        m = n * F if name == "fc1" else n * HW * HW * ch
        assert torch.equal(a[name][:m], b[name][:m]), name
        # nothing beyond the n frames is written
        assert torch.isnan(a[name][m:]).all() and torch.isnan(b[name][m:]).all(), name


@pytest.mark.gpu
@pytest.mark.parametrize("ch", [25, 32, 64])
@pytest.mark.parametrize("mode", ["bf16", "fp16", "bf16x3", "fp32"])
def test_pose_forward_batch_equals_dedicated_plan(mode, ch):
    """Remainder-packed stacked kernel (25), KC = 32 stacked kernel (32), fused paired-tap kernel (64); capacity 7,
    so n = 4 leaves a ragged remainder.  Initial state explicit, NULL (zeros) and identity."""
    cap = 7
    depth = torch.as_tensor(init.synthetic_depth(cap, seed=1, size=2 * HW)).cuda()
    h0 = torch.as_tensor(init.hidden_init((cap, HW, HW, ch), seed=5, limit=0.3)).cuda()
    big = _pose_model(mode, ch, depth)
    for n in (1, 4, 7):
        ded = _pose_model(mode, ch, depth[:n].contiguous())
        for variant in ("explicit", "zeros", "identity"):
            h = h0[:n].contiguous() if variant == "explicit" else None
            got = _pose_run(big._plan, n, depth, h, variant == "identity", ch)
            want = _pose_run(ded._plan, n, depth, h, variant == "identity", ch, batch=False)
            assert torch.equal(got[0], want[0]), (n, variant)
            assert torch.isfinite(got[0]).all()
            assert got[1] == want[1], (n, variant, got[1], want[1])
            _same_acts(got[2], want[2], n, ch)


@pytest.mark.gpu
@pytest.mark.parametrize("mode,ch", [("bf16", 25), ("bf16", 64), ("bf16x3", 32), ("fp32", 25)])
def test_stale_frames_of_a_larger_forward_do_not_leak(mode, ch):
    """A full-capacity forward on frames A, then n = 3 on frames B: fc_1's M tile rows beyond n, the operand planes
    and the chaining counters still hold A's values, and the result must be B's alone."""
    cap = 7
    A = torch.as_tensor(init.synthetic_depth(cap, seed=21, size=2 * HW, uniform=True)).cuda()
    B = torch.as_tensor(init.synthetic_depth(cap, seed=22, size=2 * HW)).cuda()
    hA = torch.as_tensor(init.hidden_init((cap, HW, HW, ch), seed=6, limit=0.5)).cuda()
    hB = torch.as_tensor(init.hidden_init((cap, HW, HW, ch), seed=7, limit=0.1)).cuda()
    big = _pose_model(mode, ch, A)
    _pose_run(big._plan, cap, A, hA, False, ch)
    got = _pose_run(big._plan, 3, B, hB[:3].contiguous(), False, ch)
    ded = _pose_model(mode, ch, B[:3].contiguous())
    want = _pose_run(ded._plan, 3, B, hB[:3].contiguous(), False, ch, batch=False)
    assert torch.equal(got[0], want[0])
    _same_acts(got[2], want[2], 3, ch)


@pytest.mark.gpu
def test_pose_forward_host_batch_chunked_upload():
    """Capacity 80: n = 33 uploads in one chunk, 70 in two, 80 in two (32-frame chunks, at most four)."""
    cap, ch, mode = 80, 25, "bf16"
    lib = _lib.load()
    depth = torch.as_tensor(init.synthetic_depth(cap, seed=4, size=2 * HW))
    dev = depth.cuda()
    host = depth.pin_memory()
    big = _pose_model(mode, ch, dev)
    _lib.check(lib.pose_set_hidden_init(big._plan, 0), "pose_set_hidden_init")
    for n in (33, 70, 80):
        out_h = torch.full((n, O), float("nan")).pin_memory()
        _lib.check(lib.pose_forward_host_batch(big._plan, n, host.data_ptr(), None, out_h.data_ptr(), _st()),
                   "pose_forward_host_batch")
        launches_h = lib.pose_plan_launch_count(big._plan)
        out_d, _, _ = _pose_run(big._plan, n, dev, None, False, ch)
        assert torch.equal(out_h, out_d.cpu()), n
        ded = _pose_model(mode, ch, dev[:n].contiguous())
        want = torch.full((n, O), float("nan")).pin_memory()
        _lib.check(lib.pose_forward_host(ded._plan, host.data_ptr(), None, want.data_ptr(), _st()),
                   "pose_forward_host")
        assert torch.equal(out_h, want), n
        assert launches_h == lib.pose_plan_launch_count(ded._plan)


def _hgru_plan(n, H, W, k, S_, T_, mode, params):
    lib = _lib.load()
    h = ctypes.c_void_p()
    _lib.check(lib.hgru_plan_create(n, H, W, k, S_, T_, _lib.MODES[mode], ctypes.byref(h)), "hgru_plan_create")
    ptrs = [params[name].data_ptr() for name in _lib.HGRU_PARAM_ORDER]
    _lib.check(lib.hgru_set_params(h, *ptrs, _st()), "hgru_set_params")
    return h


def _hgru_run(plan, n, X, O0, trace, T_, batch=True):
    lib = _lib.load()
    out = torch.full((n,) + tuple(X.shape[1:]), float("nan"), device="cuda")
    tr = [torch.full((T_, n) + tuple(X.shape[1:]), float("nan"), device="cuda") for _ in range(2)] if trace \
        else [None, None]
    if batch:
        _lib.check(lib.hgru_forward_batch(plan, n, X.data_ptr(), _ptr(O0), out.data_ptr(), _ptr(tr[0]), _ptr(tr[1]),
                                          _st()), "hgru_forward_batch")
    else:
        _lib.check(lib.hgru_forward(plan, X.data_ptr(), _ptr(O0), out.data_ptr(), _ptr(tr[0]), _ptr(tr[1]), _st()),
                   "hgru_forward")
    torch.cuda.synchronize()
    return out, tr, lib.hgru_plan_launch_count(plan)


HGRU_CASES = [("fp32", s) for s in (1, 3, 5, 7, 15)] + [("bf16", s) for s in (1, 3, 5, 7, 15)] + \
             [("bf16x3", 15), ("fp16", 15)]


@pytest.mark.gpu
@pytest.mark.parametrize("k", [25, 64])
@pytest.mark.parametrize("mode,S_", HGRU_CASES)
def test_hgru_forward_batch_equals_dedicated_plan(mode, S_, k):
    """Every filter size each mode supports, with and without H1 / H2 traces ([T, n, H, W, k]) and with a NULL
    initial state; ragged H / W."""
    cap, H, W, T_ = 5, 20, 36, 3
    lib = _lib.load()
    rng = np.random.default_rng(8)
    X = torch.as_tensor(rng.uniform(-1, 1, size=(cap, H, W, k)).astype(np.float32)).cuda()
    O0 = torch.as_tensor(init.hidden_init((cap, H, W, k), seed=3, limit=0.5)).cuda()
    params = {n: torch.as_tensor(np.asarray(v, np.float32)).cuda()
              for n, v in init.hgru_params(k, S_, T_, seed=9, stress=6.0).items()}
    big = _hgru_plan(cap, H, W, k, S_, T_, mode, params)
    try:
        for n in (1, 3, 5):
            ded = _hgru_plan(n, H, W, k, S_, T_, mode, params)
            try:
                for trace in (True, False):
                    for o0 in (O0[:n].contiguous(), None):
                        got = _hgru_run(big, n, X[:n].contiguous(), o0, trace, T_)
                        want = _hgru_run(ded, n, X[:n].contiguous(), o0, trace, T_, batch=False)
                        assert torch.equal(got[0], want[0]), (n, trace, o0 is None)
                        assert torch.isfinite(got[0]).all()
                        if trace:
                            for a, b in zip(got[1], want[1]):
                                assert torch.equal(a, b), (n, o0 is None)
                        assert got[2] == want[2]
            finally:
                lib.hgru_plan_destroy(ded)
    finally:
        lib.hgru_plan_destroy(big)


def _attn_model(depth, widths=(64, 64, 64, 64, 64), fc=64):
    am = mp.attn_model_struct()
    am.widths, am.fc_hidden = widths, fc
    am.load_params(init.attn_params(widths=widths, fc_hidden=fc, out=3, seed=8, random_bn=True))
    am.build(depth, 3)
    torch.cuda.synchronize()
    return am


@pytest.mark.gpu
@pytest.mark.parametrize("widths", [(64, 64, 64, 64, 64), (64, 128, 256, 512, 1024)])
def test_attn_forward_batch_equals_dedicated_plan(widths):
    """Odd n: the 8x8 layer puts two frames in one GEMM tile, and each layer's K split depends on n."""
    cap = 7
    lib = _lib.load()
    frames = torch.rand(cap, 120, 160, device="cuda", generator=torch.Generator("cuda").manual_seed(3))
    big = _attn_model(frames, widths)
    names = ("resized", "pool1", "pool2", "pool3", "pool4", "pool5", "fc1")
    for n in (1, 3, 5, 7):
        ded = _attn_model(frames[:n].contiguous(), widths)
        want = torch.full((n, 3), float("nan"), device="cuda")
        _lib.check(lib.attn_forward(ded._plan, frames.data_ptr(), want.data_ptr(), _st()), "attn_forward")
        want_acts = {name: ded.activation(name).reshape(-1) for name in names}
        out = torch.full((n, 3), float("nan"), device="cuda")
        _lib.check(lib.attn_forward_batch(big._plan, n, frames.data_ptr(), out.data_ptr(), _st()),
                   "attn_forward_batch")
        acts = {}
        for name in names:
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


@pytest.mark.gpu
def test_batch_out_of_range_is_rejected_with_the_capacity():
    cap, ch = 3, 25
    lib = _lib.load()
    depth = torch.as_tensor(init.synthetic_depth(cap, seed=1, size=2 * HW)).cuda()
    m = _pose_model("bf16", ch, depth)
    out = torch.zeros((cap + 1, O), device="cuda")
    host = torch.zeros((cap + 1, O)).pin_memory()
    dh = depth.cpu().pin_memory()
    frames = torch.rand(cap, 64, 64, device="cuda")
    am = _attn_model(frames)
    X = torch.rand(cap, 16, 16, 16, device="cuda")
    params = {n: torch.as_tensor(np.asarray(v, np.float32)).cuda() for n, v in init.hgru_params(16, 5, 1).items()}
    hp = _hgru_plan(cap, 16, 16, 16, 5, 1, "bf16", params)
    torch.cuda.synchronize()
    try:
        for n in (0, cap + 1, -1):
            calls = {
                "pose_forward_batch": lambda: lib.pose_forward_batch(m._plan, n, depth.data_ptr(), None,
                                                                     out.data_ptr(), _st()),
                "pose_forward_host_batch": lambda: lib.pose_forward_host_batch(m._plan, n, dh.data_ptr(), None,
                                                                               host.data_ptr(), _st()),
                "hgru_forward_batch": lambda: lib.hgru_forward_batch(hp, n, X.data_ptr(), None, X.data_ptr(), None,
                                                                     None, _st()),
                "attn_forward_batch": lambda: lib.attn_forward_batch(am._plan, n, frames.data_ptr(), out.data_ptr(),
                                                                     _st()),
            }
            for name, call in calls.items():
                assert call() == 1, (name, n)
                msg = lib.hgru_last_error().decode()
                assert name in msg and "[1, %d]" % cap in msg and "capacity" in msg, msg
        torch.cuda.synchronize()
    finally:
        lib.hgru_plan_destroy(hp)


class _Calls(object):
    """Counts the library calls named in `names` that Python makes (plan creations, parameter uploads), so that a
    test sees whether a build re-created its plan.  Handle values cannot show that: a new plan may be allocated at
    the address of the one just destroyed."""

    def __init__(self, monkeypatch, *names):
        lib = _lib.load()
        self.n = dict.fromkeys(names, 0)
        for name in names:
            def wrap(*args, _fn=getattr(lib, name), _name=name):
                self.n[_name] += 1
                return _fn(*args)
            monkeypatch.setattr(lib, name, wrap)

    def during(self, fn):
        """fn()'s result and the calls it made"""
        before = dict(self.n)
        out = fn()
        return out, {k: v - before[k] for k, v in self.n.items()}


@pytest.mark.gpu
def test_model_keeps_one_plan_below_its_capacity(monkeypatch):
    """Batches 6, 2, 6, 1 share one plan (no re-create, no set_params); each output equals a fresh model at that
    size.  Then 9 grows the plan, and 4 runs on the grown one."""
    ch, mode = 25, "bf16"
    lib = _lib.load()
    P = init.pose_params(channels=ch, S=S, T=T, hw=HW, fc_hidden=F, out=O, seed=3, stress=4.0, random_bn=True)
    depth = torch.as_tensor(init.synthetic_depth(9, seed=2, size=2 * HW)).cuda()

    def fresh():
        m = mp.model()
        m.channels, m.timesteps, m.SSF, m.SSN, m.fc_hidden, m.compute_mode = ch, T, S, S, F, mode
        m.load_params(P)      # default aux: the seeded random O_0 draw, sliced from the capacity-sized draw
        return m

    calls = _Calls(monkeypatch, "pose_plan_create", "pose_set_params")
    m = fresh()
    ws = None
    for i, n in enumerate((6, 2, 6, 1, 9, 4)):
        out, made = calls.during(lambda: m.build(depth[:n].contiguous(), O))
        want = fresh().build(depth[:n].contiguous(), O)
        torch.cuda.synchronize()
        assert torch.equal(out, want), n
        assert m.activation("hgru").shape == (n, HW, HW, ch) and m.activation("fc1").shape == (n, F)
        # the first build creates the plan; 9 replaces it by a larger one; every other size reuses it
        new = 1 if i == 0 or n == 9 else 0
        assert made == {"pose_plan_create": new, "pose_set_params": new}, (n, made)
        if n == 9:
            assert lib.pose_plan_workspace_bytes(m._plan) > ws
        elif ws is not None:
            assert lib.pose_plan_workspace_bytes(m._plan) == ws, n
        ws = lib.pose_plan_workspace_bytes(m._plan)
    assert m._plan_capacity == 9


@pytest.mark.gpu
def test_attn_model_keeps_one_plan_below_its_capacity(monkeypatch):
    lib = _lib.load()
    frames = torch.rand(9, 96, 128, device="cuda", generator=torch.Generator("cuda").manual_seed(4))
    widths = (64, 64, 64, 64, 64)
    am = mp.attn_model_struct()
    am.widths, am.fc_hidden = widths, 64
    am.load_params(init.attn_params(widths=widths, fc_hidden=64, out=3, seed=8, random_bn=True))
    calls = _Calls(monkeypatch, "attn_plan_create", "attn_set_params")
    ws = None
    for i, n in enumerate((6, 2, 6, 1, 9, 5)):
        out, made = calls.during(lambda: am.build(frames[:n].contiguous(), 3))
        want = _attn_model(frames[:n].contiguous(), widths).out_put
        assert torch.equal(out, want), n
        assert am.activation("pool5").shape == (n, 4, 4, 64)
        new = 1 if i == 0 or n == 9 else 0
        assert made == {"attn_plan_create": new, "attn_set_params": new}, (n, made)
        if n == 9:
            assert lib.attn_plan_workspace_bytes(am._plan) > ws
        ws = lib.attn_plan_workspace_bytes(am._plan)
    assert am._plan_capacity == 9


@pytest.mark.gpu
def test_contextual_circuit_reuses_a_cached_plan_with_enough_capacity(monkeypatch):
    k, S_, T_ = 16, 5, 2
    params = init.hgru_params(k, S_, T_, seed=9, stress=6.0)
    X = torch.rand(9, 24, 24, k, device="cuda", generator=torch.Generator("cuda").manual_seed(5))
    aux = dict(mp.model().aux, hidden_init="zeros")

    def run(n):
        cc = mp.ContextualCircuit(X=X[:n].contiguous(), timesteps=T_, SSN=S_, SSF=S_, aux=aux, params=params,
                                  compute_mode="bf16")
        O = cc.build(trace=True)[0]
        torch.cuda.synchronize()
        return cc, O

    seq = (6, 2, 6, 1, 9, 3)
    want = {}
    for n in sorted(set(seq)):            # each size on a plan of exactly n frames
        hm.clear_plan_cache()
        cc, O = run(n)
        want[n] = (O, cc.I_steps, cc.O_steps)
    hm.clear_plan_cache()
    calls = _Calls(monkeypatch, "hgru_plan_create", "hgru_plan_destroy")
    for i, n in enumerate(seq):
        (cc, O), made = calls.during(lambda: run(n))
        assert torch.equal(O, want[n][0]), n
        assert torch.equal(cc.I_steps, want[n][1]) and torch.equal(cc.O_steps, want[n][2]), n
        # the first build creates the plan; 9 replaces it by a larger one; every other size reuses it
        expect = {"hgru_plan_create": 1 if i == 0 or n == 9 else 0, "hgru_plan_destroy": 1 if n == 9 else 0}
        assert made == expect, (n, made)
        assert len(hm._PLAN_CACHE) == 1
        handle, capacity = next(iter(hm._PLAN_CACHE.values()))
        assert handle.value == cc._plan.value and capacity == (9 if n in (9, 3) else 6)
    hm.clear_plan_cache()


@pytest.mark.gpu
def test_streamed_forward_ragged_last_batch_keeps_the_plan(monkeypatch):
    ch, mode = 16, "bf16"
    m = mp.model()
    m.channels, m.timesteps, m.SSF, m.SSN, m.fc_hidden, m.compute_mode = ch, T, S, S, F, mode
    m.aux = dict(m.aux, hidden_init="zeros")
    m.load_params(init.pose_params(channels=ch, S=S, T=T, hw=HW, fc_hidden=F, out=O, seed=3, random_bn=True))
    batches = [torch.as_tensor(init.synthetic_depth(5, seed=30 + i, size=2 * HW)).pin_memory() for i in range(3)]
    batches.append(torch.as_tensor(init.synthetic_depth(2, seed=40, size=2 * HW)).pin_memory())
    calls = _Calls(monkeypatch, "pose_plan_create")
    got, made = calls.during(lambda: list(mp.StreamedForward(m, O)(iter(batches))))
    assert made == {"pose_plan_create": 1}          # the first batch's; the ragged last one runs on it
    assert [tuple(g.shape) for g in got] == [(5, O)] * 3 + [(2, O)]
    for g, b in zip(got, batches):
        out, made = calls.during(lambda: m.build(b, O))
        assert torch.equal(g, out) and made == {"pose_plan_create": 0}
    assert m._plan_capacity == 5


# Launches of one forward, by path: (mode, k, S) -> (per timestep, besides).  hgru_forward_batch without traces; the
# traces add two copies per timestep.  Besides the recurrence, hgru_forward_batch counts 3 and a pose forward 5 (the
# stem's three, fc_1 and the fc tail).
#   bf16 / fp16 at 15x15: the two conv launches (gates in their epilogues), + the initial-state pass
#   bf16 at S = 7: gate-in (not at t = 0: the initial-state pass makes that operand), C1, gate-out, C2
#   bf16x3 at k = 25: two launches per conv; + the initial state and the first gate-in
#   bf16x3 at k = 32: the same with the two gates as SIMT launches of every timestep
#   bf16x3 at k = 64, fp32: gate-in, C1, gate-out, C2 (fp32: + the integrations; no initial-state launch counted)
LAUNCHES = {("bf16", 25, 15): (2, 4), ("bf16", 32, 15): (2, 4), ("bf16", 64, 15): (2, 4), ("bf16", 25, 7): (4, 3),
            ("fp16", 25, 15): (2, 4), ("fp16", 64, 15): (2, 4),
            ("bf16x3", 25, 15): (4, 5), ("bf16x3", 32, 15): (6, 4), ("bf16x3", 64, 15): (4, 4),
            ("fp32", 25, 15): (6, 3)}


@pytest.mark.gpu
@pytest.mark.parametrize("T_", [1, 3])
@pytest.mark.parametrize("mode,k,S_", list(LAUNCHES))
def test_launch_counts_per_path(mode, k, S_, T_):
    """The absolute launch counts hgru_plan_launch_count and pose_plan_launch_count report, with and without the
    H1 / H2 traces (which also turn the chaining off)."""
    per_step, fixed = LAUNCHES[(mode, k, S_)]
    lib = _lib.load()
    n, H, W = 2, 20, 36
    rng = np.random.default_rng(8)
    X = torch.as_tensor(rng.uniform(-1, 1, size=(n, H, W, k)).astype(np.float32)).cuda()
    params = {name: torch.as_tensor(np.asarray(v, np.float32)).cuda()
              for name, v in init.hgru_params(k, S_, T_, seed=9).items()}
    plan = _hgru_plan(n, H, W, k, S_, T_, mode, params)
    try:
        assert _hgru_run(plan, n, X, None, False, T_)[2] == fixed + per_step * T_
        assert _hgru_run(plan, n, X, None, True, T_)[2] == fixed + (per_step + 2) * T_
    finally:
        lib.hgru_plan_destroy(plan)
    m = mp.model()
    m.channels, m.timesteps, m.SSF, m.SSN, m.fc_hidden, m.compute_mode = k, T_, S_, S_, F, mode
    m.aux = dict(m.aux, hidden_init="zeros")
    m.load_params(init.pose_params(channels=k, S=S_, T=T_, hw=HW, fc_hidden=F, out=O, seed=3, random_bn=True))
    m.build(torch.as_tensor(init.synthetic_depth(n, seed=1, size=2 * HW)).cuda(), O)
    torch.cuda.synchronize()
    assert lib.pose_plan_launch_count(m._plan) == fixed + 2 + per_step * T_
