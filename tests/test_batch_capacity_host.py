"""Host-side checks of the batch entry points (pose_forward_batch, pose_forward_host_batch, hgru_forward_batch,
attn_forward_batch) and of the initial-state draw the pose model slices for batches below its plan's capacity.
The frame-count checks against a real plan's capacity run on the GPU (tests/test_gpu_batch_capacity.py)."""
import numpy as np
import pytest

from monkey_pose_b200 import initialization as init


@pytest.mark.parametrize("n", [0, 1, 2, -1])
def test_batch_entry_points_reject_a_null_plan_before_any_cuda_call(n):
    from monkey_pose_b200 import _lib
    lib = _lib.load()
    buf = np.zeros(16, np.float32)
    calls = {
        "pose_forward_batch": lambda: lib.pose_forward_batch(None, n, buf.ctypes.data, None, buf.ctypes.data, None),
        "pose_forward_host_batch": lambda: lib.pose_forward_host_batch(None, n, buf.ctypes.data, None,
                                                                       buf.ctypes.data, None),
        "hgru_forward_batch": lambda: lib.hgru_forward_batch(None, n, buf.ctypes.data, None, buf.ctypes.data, None,
                                                             None, None),
        "attn_forward_batch": lambda: lib.attn_forward_batch(None, n, buf.ctypes.data, buf.ctypes.data, None),
    }
    for name, call in calls.items():
        assert call() == 1, name                                      # HGRU_E_INVALID
        assert lib.hgru_last_error().decode() == name + ": null plan"


@pytest.mark.parametrize("shape", [(7, 4, 4, 3), (256, 8, 8, 25), (9, 64, 64, 2)])
def test_initial_state_draw_of_n_frames_is_a_slice_of_the_draw_at_capacity(shape):
    """model.build draws the seeded O_0 once at its plan's capacity and slices [:n]: numpy's Generator.uniform fills
    in C order, so the slice is bit for bit the draw of n frames."""
    N = shape[0]
    full = init.hidden_init(shape, seed=49)
    for n in sorted({1, 2, N // 2, N - 1, N} - {0}):
        part = init.hidden_init((n,) + shape[1:], seed=49)
        assert np.array_equal(part.view(np.uint32), full[:n].view(np.uint32)), n
