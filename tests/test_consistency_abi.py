"""CPU-side checks of the filter-consistency surface: the new entry points refuse null handles before any device work,
fleet.consistency's chi-square intervals match scipy, and the numpy m2 the GPU tests compare the captured NIS against
is the distance the CPU oracle's gate decides on."""
import ctypes as C

import numpy as np
import pytest
from scipy.stats import chi2

import consistency_ref as cref
import np_ref
from slam_localization_b200 import engine, fleet, synth


def test_entry_points_refuse_null_handles():
    L = engine.lib()
    out = (C.c_double * 6)()
    assert L.slb_set_nis_capture(None, 1) == -1
    assert L.slb_consistency_stats(None, None, 0, 0, None, out, None) == -1
    assert L.slb_gather_consistency(None, None, None, 0, 0, None, out, None) == -1
    assert L.slb_device_ptr(None, engine.FIELD_NIS, C.byref(C.c_void_p())) == -1
    assert L.slb_download(None, engine.FIELD_NIS, out, 6, None) == -1


def test_facade_header_declares_the_new_members():
    import os
    hdr = open(os.path.join(os.path.dirname(os.path.abspath(np_ref.__file__)), "..", "slam-localization_b200", "facade",
                            "localization_b200.hpp")).read()
    for name in ("setNisCapture", "mahalanobis", "consistencyStats"):
        assert name in hdr


@pytest.mark.parametrize("k", [300, 301, 1000, 9 * 65536, 3 * 203 * 50])
@pytest.mark.parametrize("p", [0.9, 0.95, 0.99])
def test_chi2_interval_matches_scipy(k, p):
    m = 100
    s = [0, 0, 0, m, m * 1.0, 0]
    r = fleet.consistency(s, 1, k / m, p=p)
    lo, hi = r["anis_interval"]
    np.testing.assert_allclose(lo * m, chi2.ppf((1 - p) / 2, k), rtol=1e-3)
    np.testing.assert_allclose(hi * m, chi2.ppf((1 + p) / 2, k), rtol=1e-3)


def test_consistency_hand_worked():
    # two steps of 100 instances, NEES over 3 dof, NIS over 3 dof
    a = [100, 310.0, 1500.0, 100, 290.0, 1200.0]
    b = [100, 290.0, 1400.0, 50, 160.0, 800.0]
    r = fleet.consistency([a, b], nees_dof=3, nis_dof=3, p=0.95)
    assert r["anees_count"] == 200 and r["anis_count"] == 150
    assert r["anees"] == 600.0 / 200 and r["anis"] == 450.0 / 150
    # Wilson-Hilferty by hand for M d = 600, p = 0.975: z = 1.959963984540054, h = 2 / 5400
    h = 2.0 / 5400.0
    want = 600.0 * (1 - h + 1.959963984540054 * np.sqrt(h)) ** 3 / 200
    assert abs(r["anees_interval"][1] - want) <= 1e-12 * want
    assert r["anees_interval"][0] < 3.0 < r["anees_interval"][1]
    empty = fleet.consistency(np.zeros(6), 3, 3)
    assert empty["anees_count"] == 0 and np.isnan(empty["anees"]) and empty["anees_interval"] is None
    with pytest.raises(ValueError):
        fleet.consistency(np.zeros(5), 3, 3)


def _gate_rejects(st):
    return (st & engine.ST_GATE_REJECT) != 0


def test_numpy_m2_is_what_the_oracle_gate_decides_on_usckf(slo):
    for nk, nl in [(3, 9), (6, 6), (9, 3)]:
        B = 24
        sc = synth.usckf_scenario(B, seed=501 + nk, nk=nk, nl=nl)
        sc["z"] = sc["z"] + 0.15
        m2 = np.array([cref.usckf_m2(nk, sc["mu"][i], sc["P"][i], sc["z"][i], sc["R"]) for i in range(B)])
        _, _, st, _ = slo.usckf_step(slo.PM_USCKF_TEST, slo.MM_USCKF_VO, nk, nl, sc["mu"], sc["P"], None, 0.0, None, sc["z"],
                                     sc["R"], gate_dof=nk, predict=False)
        th = cref.CHI2_5[nk]
        np.testing.assert_array_equal(_gate_rejects(st), m2 >= th)
        assert _gate_rejects(st).any() and not _gate_rejects(st).all()
    # and the numpy distance agrees with the scipy-based restatement's S and innovation
    i = 3
    mu, P, z, R = sc["mu"][i], sc["P"][i], sc["z"][i], sc["R"]
    X = np_ref.sigma_points(np_ref.AUG_BLOCKS, mu, np.zeros(P.shape[0]), P, nk + nl)
    Z = np.array([np_ref.mm_usckf_vo(x, nk) for x in X])
    zb = Z.mean(axis=0)
    S = 0.5 * (Z - zb).T @ (Z - zb) + R
    want = (z - zb) @ np.linalg.solve(S, z - zb)
    assert abs(cref.usckf_m2(nk, mu, P, z, R) - want) <= 1e-10 * want


def test_numpy_m2_is_what_the_oracle_gate_decides_on_ukfom(slo):
    for layout in (9, 6):
        B = 64
        sc = synth.ukfom_scenario(B, seed=511, layout=layout)
        sc["z"] = sc["z"] + 0.03
        m2 = np.array([cref.ukf_m2(sc["mu"][i], sc["P"][i], sc["z"][i], sc["R"]) for i in range(B)])
        _, _, st, _ = slo.ukf_step(layout, slo.PM_UKFOM_IMU if layout == 9 else slo.PM_POSE6_ODOM, slo.MM_GPS_POS, sc["mu"],
                                   sc["P"], None, 0.0, None, sc["z"], sc["R"], gate_dof=3, predict=False)
        np.testing.assert_array_equal(_gate_rejects(st), m2 >= cref.CHI2_5[3])
        assert _gate_rejects(st).any() and not _gate_rejects(st).all()


def test_numpy_nees_restatement_on_a_known_draw():
    rng = np.random.default_rng(521)
    blocks, nf, B = [0, 1, 0] * 4, 5, 16
    n = 3 * len(blocks) + nf
    mu = synth.random_q(rng, B, blocks, nfeat=nf)
    P = synth.random_spd(rng, B, n, 1e-2, 1e2)
    w = rng.normal(size=(B, n))
    truth = cref.boxplus(blocks, nf, mu, np.einsum("bij,bj->bi", np.linalg.cholesky(P), w))
    np.testing.assert_allclose(cref.nees(blocks, nf, truth, mu, P, 0, n), (w * w).sum(axis=1), rtol=1e-9)
