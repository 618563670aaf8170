"""The USCKF predict runs in two kernels: alone (slb_usckf_predict: predict12_kernel on the rows it touches) and inside
the fused step (usckf_step_kernel, on the resident record).  Both run the same predict body, so predict() followed by
update() must give the fused step()'s results bit for bit, for every built shape and with shared or per-instance Q."""
import numpy as np
import pytest

from slam_localization_b200 import engine, synth

pytestmark = pytest.mark.gpu
B = 203                  # ragged against the 8-warp predict CTAs and the 4- / 6-warp step CTAs
SHAPES = [(3, 0), (3, 3), (3, 6), (3, 9), (6, 0), (6, 3), (6, 6), (9, 0), (9, 3)]


@pytest.mark.parametrize("per_instance_q", [False, True])
@pytest.mark.parametrize("nk,nl", SHAPES)
def test_usckf_predict_then_update_is_bitwise_the_fused_step(nk, nl, per_instance_q):
    sc = synth.usckf_scenario(B, seed=251, nk=nk, nl=nl)
    Q = sc["Q"]
    if per_instance_q:
        rng = np.random.default_rng(252)
        Q = synth.random_spd(rng, B, 12, 1.0, 10.0) * np.abs(np.diag(sc["Q"])).mean()
    two = engine.Usckf(B, nk=nk, nl=nl)
    two.set_state(sc["mu"], sc["P"])
    two.predict(engine.PM_USCKF_TEST, sc["u"], sc["dt"], Q)
    two.update(engine.MM_USCKF_VO, sc["z"], sc["R"])
    one = engine.Usckf(B, nk=nk, nl=nl)
    one.set_state(sc["mu"], sc["P"])
    one.step(engine.PM_USCKF_TEST, engine.MM_USCKF_VO, sc["u"], sc["dt"], Q, sc["z"], sc["R"])
    np.testing.assert_array_equal(two.mu(), one.mu())
    np.testing.assert_array_equal(two.P(), one.P())
    np.testing.assert_array_equal(two.status(), one.status())
    assert not one.status().any()
