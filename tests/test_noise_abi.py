"""CPU-side checks of the per-instance noise layout (slb_set_noise_layout): the entry point validates its handle before
touching a device, and the engine decides the layout from the shapes of Q / R, refusing any other shape before the
library is called."""
import ctypes as C

import numpy as np
import pytest

from slam_localization_b200 import engine


def test_set_noise_layout_rejects_a_null_handle_without_a_gpu():
    L = engine.lib()
    assert L.slb_set_noise_layout(None, engine.NOISE_Q_PER_INSTANCE) == -1
    assert b"slb_set_noise_layout" in L.slb_last_error()
    assert L.slb_set_noise_layout(None, 0) == -1


class _Fake(engine.Batch):
    """The engine's shape logic without a device: set_noise_layout only records the flags."""

    def __init__(self, B):
        self.B, self.noise, self.h, self.calls = B, 0, C.c_void_p(), []

    def set_noise_layout(self, flags):
        self.calls.append(flags)
        self.noise = flags


def test_engine_decides_the_noise_layout_from_shapes():
    f = _Fake(5)
    f._use_noise(Q=np.eye(12), n=12)
    assert f.calls == []                                     # shared: the default layout, no library call
    f._use_noise(Q=np.zeros((5, 12, 12)), n=12)
    assert f.calls == [engine.NOISE_Q_PER_INSTANCE]
    f._use_noise(R=np.zeros((5, 3, 3)), m=3)                 # the Q bit is kept
    assert f.noise == engine.NOISE_Q_PER_INSTANCE | engine.NOISE_R_PER_INSTANCE
    f._use_noise(Q=np.eye(12), n=12, R=np.zeros((5, 3, 3)), m=3)
    assert f.noise == engine.NOISE_R_PER_INSTANCE
    n = len(f.calls)
    f._use_noise(Q=np.eye(12), n=12, R=np.zeros((5, 3, 3)), m=3)
    assert len(f.calls) == n                                 # unchanged layout: cached on the batch
    f._use_noise(R=np.eye(3), m=3)
    assert f.noise == 0


@pytest.mark.parametrize("shape", [(12,), (144,), (12, 11), (4, 12, 12), (6, 12, 12), (5, 12, 11), (1, 5, 12, 12)])
def test_engine_rejects_malformed_noise_shapes(shape):
    f = _Fake(5)
    with pytest.raises(ValueError, match="shape"):
        f._use_noise(Q=np.zeros(shape), n=12)
    assert f.calls == []


def test_engine_step_host_refuses_per_instance_noise():
    f = _Fake(5)
    with pytest.raises(ValueError, match="step_host"):
        f._host_noise(np.zeros((5, 12, 12)), 12, np.eye(3), 3)
    with pytest.raises(ValueError, match="step_host"):
        f._host_noise(np.eye(12), 12, np.zeros((5, 3, 3)), 3)
    with pytest.raises(ValueError, match="step_host"):
        f._host_noise(np.zeros(5 * 144), 12, np.eye(3), 3)   # flat, but one matrix per instance
    f._host_noise(np.eye(12).ravel(), 12, np.eye(3), 3)      # a flat shared matrix passes as it did before
    f.noise = engine.NOISE_R_PER_INSTANCE                    # shared arrays restore the shared layout
    f._host_noise(np.eye(12), 12, np.eye(3), 3)
    assert f.noise == 0
