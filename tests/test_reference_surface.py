"""CPU: every function and method the reference defines in the files of the hot path and its neighbouring stages has a
same-named counterpart in the mirror package -- as a kernel-backed method, or (for what SURVEY.md section 8 row a19
lists as declared but not on the configured path) as a method that raises the reference's own NotImplementedError.  The
few names left out are listed here with the reason.  The reference's names are stored in golden/reference_surface.json;
with MONKEY_POSE_REFERENCE naming a checkout of the reference (krg-nandu/monkey-pose) they are also read from its source,
the stored ones must be among them, and the tests use the names read."""
import json
import os
import sys

import pytest
import torch

import monkey_pose_b200 as mp
from monkey_pose_b200 import pose_evaluation, tf_monkeydetector

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
sys.path.insert(0, GOLDEN)
import make_golden_reference_surface as surface  # noqa: E402

STORED = json.load(open(os.path.join(GOLDEN, "reference_surface.json")))
REF = os.environ.get("MONKEY_POSE_REFERENCE", "")


def _defs(path, cls=None):
    """Names the reference defines at module level (cls None) or inside class `cls` of `path`."""
    names = list(STORED[path][cls or ""])
    if os.path.isdir(REF):
        read = list(surface.defs(open(os.path.join(REF, path)).read(), cls or ""))
        assert set(names) <= set(read), (path, cls, sorted(set(names) - set(read)))
        names = read
    return names


def test_contextual_circuit_surface():
    names = _defs("hgru_module.py", "ContextualCircuit")
    assert len(names) >= 25
    missing = [n for n in names if not hasattr(mp.ContextualCircuit, n)]
    assert not missing, missing
    assert "auxilliary_variables" in _defs("hgru_module.py") and hasattr(mp.hgru_module, "auxilliary_variables")
    # the off-path methods raise the reference's error type
    cc = mp.ContextualCircuit(X=torch.zeros(1, 8, 8, 4), timesteps=2, SRF=1, SSN=15, SSF=15, aux=mp.model().aux)
    for n, args in (("apply_tuning", (None, "P")), ("zoneout", (0.5,)), ("hierarchical_convolutions", (None, "p_r", None)),
                    ("mely_input_integration", (None,) * 4), ("mely_output_integration", (None,) * 4),
                    ("input_integration_control", (None,) * 4), ("output_integration_control", (None,) * 4)):
        with pytest.raises(NotImplementedError):
            getattr(cc, n)(*args)
    assert cc.symmetric_weights is True          # as in the reference, the option shadows the method of that name


def test_pose_model_and_attention_model_surface():
    for path, cls, mirror in (("hgru_pose.py", "model", mp.model),
                              ("train_cnn_networks_hgru.py", "attn_model_struct", mp.attn_model_struct)):
        names = _defs(path, cls)
        assert "build" in names and "conv_layer" in names
        missing = [n for n in names if not hasattr(mirror, n)]
        assert not missing, (cls, missing)


def test_detector_surface():
    names = _defs("tf_monkeydetector.py", "tfMonkeyDetector")
    # checkImage / getNDValue read self.dpt, which the reference's constructor no longer sets (and getNDValue opens a
    # debugger): they cannot run in the reference either
    left_out = {"checkImage", "getNDValue"}
    missing = [n for n in names if n not in left_out and not hasattr(tf_monkeydetector.tfMonkeyDetector, n)]
    assert not missing, missing
    assert left_out <= set(names)


def test_metric_file_surface():
    names = _defs("pose_evaluation.py")
    left_out = {"main"}                           # the plotting script of the file (:94-209)
    missing = [n for n in names if n not in left_out and not hasattr(pose_evaluation, n)]
    assert not missing, missing
    assert len([n for n in names if n not in left_out]) == 10


def test_data_stage_functions_of_the_trainer():
    names = _defs("train_cnn_networks_hgru.py")
    assert "prepare_data" in names and "prepare_data_test" in names
    assert hasattr(tf_monkeydetector, "prepare_data") and hasattr(tf_monkeydetector, "prepare_data_test")
