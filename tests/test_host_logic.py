"""CPU: host-side mirror of the reference interface -- option handling, error behaviour, parameter
shapes, sharding arithmetic.  (No kernels run here.)"""
import os

import numpy as np
import pytest
import torch

import monkey_pose_b200 as mp
from monkey_pose_b200 import initialization as init
from monkey_pose_b200.sharding import shard_bounds

POSE_AUX = mp.model().aux


def _cc(**kw):
    aux = dict(POSE_AUX)
    aux.update(kw.pop("aux", {}))
    return mp.ContextualCircuit(X=torch.zeros(2, 8, 8, 8), timesteps=3, SRF=1, SSN=15, SSF=15, aux=aux, **kw)


def test_constructor_mirrors_reference_attributes():
    cc = _cc()
    assert (cc.n, cc.h, cc.w, cc.k) == (2, 8, 8, 8)
    assert cc.SSF_ext == 15 and cc.p_shape == [15, 15, 8, 8]
    assert cc.i_shape == [1, 1, 8, 8] and cc.bias_shape == [1, 1, 1, 8]
    assert cc["timesteps"] == 3 and "gru_gates" in cc            # __getitem__ / __contains__ sugar
    assert cc.gru_gates is True and cc.return_weights is True     # aux merged over the defaults
    assert mp.ContextualCircuit(X=torch.zeros(1, 4, 4, 4), SSF=28, aux=POSE_AUX).SSF_ext == 29


def test_aux_defaults_match_reference_keys():
    d = mp.auxilliary_variables()
    for k in ("lesions", "return_weights", "hidden_init", "gate_bias_init", "gru_gates", "integration_type",
              "multiplicative_excitation", "adapation", "rectify_weights", "store_states"):
        assert k in d
    assert d["gru_gates"] is False and d["integration_type"] == "alternate" and d["hidden_init"] == "random"


@pytest.mark.parametrize("aux", [
    {"integration_type": "mely"}, {"integration_type": "control"}, {"integration_type": "bogus"},
    {"recurrent_nl": "relu"}, {"recurrent_nl": "bogus"}, {"gru_gates": False}, {"output_gru_gates": True},
    {"multiplicative_excitation": False}, {"rectify_weights": True}, {"atrous_convolutions": 2},
    {"gate_filter": 3}, {"lesions": ["P"]}, {"store_states": True}, {"dropout": 0.5},
])
def test_off_path_options_raise_not_implemented(aux):
    with pytest.raises(NotImplementedError):
        _cc(aux=aux)


def test_list_ssf_and_strides_raise():
    with pytest.raises(NotImplementedError):
        mp.ContextualCircuit(X=torch.zeros(1, 4, 4, 4), SSF=[3, 5], aux=POSE_AUX)
    with pytest.raises(NotImplementedError):
        mp.ContextualCircuit(X=torch.zeros(1, 4, 4, 4), SSF=5, strides=[1, 2, 2, 1], aux=POSE_AUX)


def test_build_without_cuda_fails_loudly():
    if torch.cuda.is_available():
        pytest.skip("CPU-only check")
    with pytest.raises(RuntimeError):
        _cc().build()


def test_model_defaults_are_the_references():
    m = mp.model()
    assert (m.SRF, m.SSN, m.SSF, m.timesteps, m.padding) == (1, 15, 15, 8, 'SAME')
    assert m._BATCH_NORM_DECAY == 0.997 and m._BATCH_NORM_EPSILON == 1e-5
    assert m.aux["gru_gates"] and m.aux["adapation"] and m.aux["recurrent_nl"] == "tanh"
    assert m["timesteps"] == 8 and "aux" in m
    with pytest.raises(RuntimeError, match="CUDA"):          # the layer-wise training-mode forward has no CPU fallback
        m.build(torch.zeros(1, 128, 128, 1), 69, train_mode=True)
    with pytest.raises(ValueError):
        m.build(torch.zeros(1, 128, 64, 1), 69)
    for meth in ("conv_layer", "max_pool", "fc_layer", "hgru_layer", "get_conv_var", "get_fc_var", "get_var"):
        assert callable(getattr(m, meth))                    # hgru_pose.py:107-216
    with pytest.raises(AttributeError):
        m.conv1                                              # set by build(), as in the reference


def test_param_generators_shapes_and_statistics():
    p = init.hgru_params(64, 15, 8, seed=1)
    assert p["p_r"].shape == (15, 15, 64, 64) and p["rho"].shape == (8,)
    lim = np.sqrt(6.0 / (225 * 64 + 225 * 64))
    assert abs(np.abs(p["p_r"]).max() - lim) < 1e-3 * lim + 1e-6        # xavier-uniform limit 0.01443
    assert np.all(p["i_b"] <= 0) and np.allclose(p["o_b"], -p["i_b"])   # chronos: -log U(1, T-1)
    assert np.all(p["rho"] == 1)
    P = init.pose_params(channels=8, hw=8, fc_hidden=16, out=6)
    assert P["fc_1/fc_1_weights"].shape == (8 * 8 * 8, 16)
    assert P["batch_normalization_4/gamma"].shape == (16,)
    d = init.synthetic_depth(3, seed=0)
    assert d.shape == (3, 128, 128, 1) and d.min() >= 0 and d.max() <= 1 and (d == 1.0).mean() > 0.2


def test_shard_bounds_partition_the_batch():
    for n, w in ((4096, 8), (256, 1), (10, 4), (3, 8)):
        spans = [shard_bounds(n, r, w) for r in range(w)]
        assert spans[0][0] == 0 and spans[-1][1] == n
        assert all(a[1] == b[0] for a, b in zip(spans, spans[1:]))
        assert max(h - l for l, h in spans) - min(h - l for l, h in spans) <= 1


def test_crop_windows_batch_equals_per_frame_reference_arithmetic():
    """tfMonkeyDetector._windows_batch (array form used at batch size) == the line-by-line mirror of
    comToBounds / cropArea3D's window arithmetic (tf_monkeydetector.py:193-206, 309-362) for every frame."""
    import numpy as np
    from monkey_pose_b200 import tf_monkeydetector as tmd
    md = tmd.tfMonkeyDetector(365.456, 365.456, 256, 212, [800, 800, 1200], 200, 10000)
    rng = np.random.default_rng(0)
    n = 500
    coms = np.stack([rng.uniform(0.1, 1.1, n) * 424, rng.uniform(0.1, 0.75, n) * 512,
                     rng.uniform(0.08, 0.35, n) * 10000], 1)
    ints, z, Ms = md._windows_batch(coms, 424, 512, (128, 128))
    for i in range(n):
        a, b, M = md._window(coms[i], 424, 512, (128, 128))
        assert tuple(int(v) for v in ints[i]) == tuple(int(v) for v in a)
        assert np.array_equal(z[i], np.asarray(b, np.float32))
        np.testing.assert_allclose(Ms[i], M, rtol=0, atol=1e-12)


def test_bench_has_no_rank_conditional_steps():
    """Every rank must run the same sequence of steps (each multi-GPU step ends in an all-gather): a forward
    pass under `if clocks:` / `if rank == 0:` deadlocks torchrun runs.  Static check of bench.py."""
    import ast
    import os
    src = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "bench.py")).read()
    tree = ast.parse(src)
    bad = []
    for node in ast.walk(tree):
        if not isinstance(node, ast.If):
            continue
        names = {n.id for n in ast.walk(node.test) if isinstance(n, ast.Name)}
        if not names & {"rank", "clocks"}:
            continue
        for sub in node.body + node.orelse:
            for call in ast.walk(sub):
                if isinstance(call, ast.Call) and isinstance(call.func, ast.Name) and \
                        call.func.id in ("step_dev", "step_host", "timed", "gather_predictions", "PredictionGatherer"):
                    bad.append((node.lineno, call.func.id))
    assert not bad, bad


def test_product_build_defines_no_development_switch():
    """The kernels carry compile-time development switches (HGRU_DBG_*, HGRU_STACK_*) for the devtools' A/B builds;
    the library's Makefile must not define any of them, and every switch that exists is off by default (#ifdef)."""
    import os
    import re
    csrc = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "monkey-pose_b200", "csrc")
    mk = open(os.path.join(csrc, "Makefile")).read()
    assert "-DHGRU_" not in mk
    switches = set()
    for fn in os.listdir(csrc):
        if fn.endswith((".cuh", ".cu", ".inl")):
            src = open(os.path.join(csrc, fn)).read()
            switches |= set(re.findall(r"#\s*ifn?def\s+(HGRU_(?:DBG|STACK)_\w+)", src))
            for name in re.findall(r"#\s*define\s+(HGRU_(?:DBG|STACK)_\w+)", src):
                assert name == "HGRU_STACK_EPI", (fn, name)      # (a local helper macro, not a switch)
    assert {"HGRU_STACK_NO_REM", "HGRU_STACK_NGRP4", "HGRU_DBG_NO_GLOBAL"} <= switches


def test_library_reads_only_the_chaining_switch_from_the_environment():
    """The one run-time switch of the library is HGRU_NO_CHAIN=1 (plain stream order between the conv launches, the
    reference order of the chaining test).  Every getenv() argument in the library's sources (not the devtools) is
    collected, a non-literal one as its expression, so a switch read through a helper is caught too."""
    import os
    import re
    csrc = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "monkey-pose_b200", "csrc")
    names = set()
    for root, dirs, files in os.walk(csrc):
        dirs[:] = [d for d in dirs if d != "devtools"]
        for fn in files:
            if fn.endswith((".cu", ".cuh", ".inl", ".h", ".cpp")):
                src = open(os.path.join(root, fn)).read()
                names |= {a.strip().strip('"') for a in re.findall(r"\bgetenv\(([^)]*)\)", src)}
    assert names == {"HGRU_NO_CHAIN"}


def test_circuit_step_methods_mirror_the_reference_signatures():
    """ContextualCircuit exposes the reference's per-timestep methods (hgru_module.py:505-861) with the same argument
    names and order; they need CUDA tensors (no CPU fallback)."""
    import inspect
    import re
    ref_path = os.path.join(os.environ.get("MONKEY_POSE_REFERENCE", ""), "hgru_module.py")
    src = open(ref_path).read() if os.path.isfile(ref_path) else None
    want = {
        "conv_2d_op": ["self", "data", "weight_key", "out_key", "weights", "symmetric_weights", "rectify"],
        "p_convolution": ["self", "data", "key", "rectification"],
        "process_p": ["self", "data", "key", "rectification", "full"],
        "circuit_input": ["self", "O"],
        "circuit_output": ["self", "I"],
        "input_integration": ["self", "P", "I", "O", "I_update"],
        "output_integration": ["self", "P", "I", "O", "O_update"],
        "full": ["self", "i0", "O", "I", "store_O", "store_I"],
        "condition": ["self", "i0", "O", "I", "store_I", "store_O"],
    }
    for name, args in want.items():
        got = [a for a in inspect.signature(getattr(mp.ContextualCircuit, name)).parameters if not a.startswith("_")]
        assert got == args, (name, got)
        if src is not None:                      # with the reference's source: the table above IS the reference's
            m = re.search(r"def %s\(([^)]*)\)" % name, src)
            ref = [a.split("=")[0].strip() for a in m.group(1).replace("\n", " ").split(",") if a.strip()]
            assert ref == args, (name, ref)
    cc = mp.ContextualCircuit(X=torch.zeros(1, 8, 8, 4), timesteps=2, SRF=1, SSN=15, SSF=15, aux=mp.model().aux)
    assert cc.condition(0, None, None, None, None) and not cc.condition(2, None, None, None, None)
    with pytest.raises(RuntimeError):
        cc.k = 4
        cc.lateral_bias = torch.zeros(1, 1, 1, 4)
        cc.p_r = torch.zeros(15, 15, 4, 4)
        cc.process_p(torch.zeros(1, 8, 8, 4), "p_r", None)          # host tensor: fails loudly
