"""Per-instance process and measurement noise (slb_set_noise_layout) for the UKFoM, USCKF and MSCKF-predict batches.

A batch of B stands for B reference objects that were handed different covariances.  The per-instance kernels change
only the address a noise entry is read from, so B copies of the shared matrix must give the shared path's results bit
for bit; distinct matrices are checked against the CPU oracle called once per instance with that instance's Q / R."""
import ctypes as C

import numpy as np
import pytest

import parity
from slam_localization_b200 import engine, synth

pytestmark = pytest.mark.gpu
B = 203                  # ragged against the 8-instance UKF warps and the 4- / 6-warp USCKF CTAs
AUG = synth.STATE_BLOCKS * 3
MODES = ["predict", "update", "step"]
UKF_CASES = [(9, engine.PM_UKFOM_IMU), (6, engine.PM_POSE6_ODOM)]
USCKF_SHAPES = [(3, 9), (3, 0), (6, 6), (9, 3)]


def _spd(rng, n, base):
    """B random SPD n x n matrices whose scales spread over two decades around `base`."""
    return synth.random_spd(rng, B, n, 1.0, 10.0) * (base * 10.0 ** rng.uniform(-1, 1, size=(B, 1, 1)))


def _rep(M):
    return np.ascontiguousarray(np.broadcast_to(M, (B,) + M.shape))


# ---- UKFoM --------------------------------------------------------------------------------------------------------
def _ukf(layout, pm, mode, sc, Q, R, gate=0):
    f = engine.Ukf(B, layout=layout)
    f.set_state(sc["mu"], sc["P"])
    if mode == "predict":
        f.predict(pm, sc["u"], sc["dt"], Q)
    elif mode == "update":
        f.update(engine.MM_GPS_POS, sc["z"], R, gate_dof=gate)
    else:
        f.step(pm, engine.MM_GPS_POS, sc["u"], sc["dt"], Q, sc["z"], R, gate_dof=gate)
    return f.mu(), f.P(), f.status()


def _ukf_oracle(slo, layout, pm, mode, sc, Q, R, gate=0, only=None):
    out = []
    for i in range(B) if only is None else only:
        s = slice(i, i + 1)
        mu, P, st, _ = slo.ukf_step(layout, pm, slo.MM_GPS_POS, sc["mu"][s], sc["P"][s], sc["u"][s], sc["dt"], Q[i], sc["z"][s],
                                    R[i], gate_dof=gate, predict=mode != "update", update=mode != "predict")
        out.append((mu[0], P[0], st[0]))
    return [np.array(x) for x in zip(*out)]


def _ukf_noise(sc, layout, seed):
    rng = np.random.default_rng(seed)
    return _spd(rng, layout, np.abs(np.diag(sc["Q"])).mean()), _spd(rng, 3, sc["R"][0, 0])


@pytest.mark.parametrize("layout,pm", UKF_CASES)
@pytest.mark.parametrize("mode", MODES)
def test_ukf_replicated_noise_is_bitwise_the_shared_path(layout, pm, mode):
    sc = synth.ukfom_scenario(B, seed=201, layout=layout)
    a = _ukf(layout, pm, mode, sc, sc["Q"], sc["R"])
    b = _ukf(layout, pm, mode, sc, _rep(sc["Q"]), _rep(sc["R"]))
    for x, y in zip(a, b):
        np.testing.assert_array_equal(x, y)
    assert not a[2].any()


@pytest.mark.parametrize("layout,pm", UKF_CASES)
@pytest.mark.parametrize("mode", MODES)
def test_ukf_distinct_noise_matches_the_oracle_per_instance(slo, layout, pm, mode):
    sc = synth.ukfom_scenario(B, seed=202, layout=layout)
    Q, R = _ukf_noise(sc, layout, 203)
    mu, P, st = _ukf(layout, pm, mode, sc, Q, R)
    mu_r, P_r, st_r = _ukf_oracle(slo, layout, pm, mode, sc, Q, R)
    assert not st.any() and not st_r.any()
    parity.assert_parity(slo, synth.LAYOUT_BLOCKS[layout], mu, P, mu_r, P_r)
    shared = _ukf(layout, pm, mode, sc, Q[0], R[0])   # the noise did reach every instance
    assert not np.array_equal(P[1:], shared[1][1:])


# ---- USCKF --------------------------------------------------------------------------------------------------------
def _usckf(nk, nl, mode, sc, Q, R, gate=0):
    f = engine.Usckf(B, nk=nk, nl=nl)
    f.set_state(sc["mu"], sc["P"])
    if mode == "predict":
        f.predict(engine.PM_USCKF_TEST, sc["u"], sc["dt"], Q)
    elif mode == "update":
        f.update(engine.MM_USCKF_VO, sc["z"], R, gate_dof=gate)
    else:
        f.step(engine.PM_USCKF_TEST, engine.MM_USCKF_VO, sc["u"], sc["dt"], Q, sc["z"], R, gate_dof=gate)
    return f.mu(), f.P(), f.status()


def _usckf_oracle(slo, nk, nl, mode, sc, Q, R, gate=0, only=None):
    out = []
    for i in range(B) if only is None else only:
        s = slice(i, i + 1)
        mu, P, st, _ = slo.usckf_step(slo.PM_USCKF_TEST, slo.MM_USCKF_VO, nk, nl, sc["mu"][s], sc["P"][s], sc["u"][s], sc["dt"],
                                      Q[i], sc["z"][s], R[i], gate_dof=gate, predict=mode != "update",
                                      update=mode != "predict")
        out.append((mu[0], parity.symmetrize_lower(P)[0], st[0]))
    return [np.array(x) for x in zip(*out)]


def _usckf_noise(sc, nk, seed):
    rng = np.random.default_rng(seed)
    return _spd(rng, 12, np.abs(np.diag(sc["Q"])).mean()), _spd(rng, nk, sc["R"][0, 0])


@pytest.mark.parametrize("nk,nl", USCKF_SHAPES)
@pytest.mark.parametrize("mode", MODES)
def test_usckf_replicated_noise_is_bitwise_the_shared_path(nk, nl, mode):
    sc = synth.usckf_scenario(B, seed=211, nk=nk, nl=nl)
    a = _usckf(nk, nl, mode, sc, sc["Q"], sc["R"])
    b = _usckf(nk, nl, mode, sc, _rep(sc["Q"]), _rep(sc["R"]))
    for x, y in zip(a, b):
        np.testing.assert_array_equal(x, y)
    assert not a[2].any()


@pytest.mark.parametrize("nk,nl", USCKF_SHAPES)
@pytest.mark.parametrize("mode", MODES)
def test_usckf_distinct_noise_matches_the_oracle_per_instance(slo, nk, nl, mode):
    sc = synth.usckf_scenario(B, seed=212, nk=nk, nl=nl)
    Q, R = _usckf_noise(sc, nk, 213)
    mu, P, st = _usckf(nk, nl, mode, sc, Q, R)
    mu_r, P_r, st_r = _usckf_oracle(slo, nk, nl, mode, sc, Q, R)
    assert not st.any() and not st_r.any()
    parity.assert_parity(slo, AUG, mu, P, mu_r, P_r, nfeat=nk + nl)
    shared = _usckf(nk, nl, mode, sc, Q[0], R[0])
    assert not np.array_equal(P[1:], shared[1][1:])


@pytest.mark.parametrize("mode", [engine.STATEK, engine.STATEK_L])
def test_usckf_set_measurement_per_instance_noise(slo, mode):
    sc = synth.usckf_scenario(B, seed=221)
    ln = 3 if mode == engine.STATEK else 9
    rng = np.random.default_rng(222)
    z = rng.normal(size=(B, ln))
    R = _spd(rng, ln, 0.01)

    def run(Rx):
        f = engine.Usckf(B)
        f.set_state(sc["mu"], sc["P"])
        f.set_measurement(mode, z, Rx)
        return f.mu(), f.P()

    for x, y in zip(run(R[5]), run(_rep(R[5]))):           # replicated == shared, bitwise
        np.testing.assert_array_equal(x, y)
    mu, P = run(R)
    for i in range(B):                                     # a pure copy: exactly the oracle's, instance by instance
        mo, Po = slo.usckf_set_measurement(mode, 3, 9, sc["mu"][i:i + 1], sc["P"][i:i + 1], z[i:i + 1], R[i])
        np.testing.assert_array_equal(mu[i], mo[0])
        np.testing.assert_array_equal(P[i], parity.symmetrize_lower(Po)[0])


# ---- MSCKF predict ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("pm", [engine.PM_MSCKF_DELTAPOSE, engine.PM_USCKF_TEST])
def test_msckf_predict_per_instance_q(slo, pm):
    k = 10
    sc = synth.msckf_scenario(B, seed=231, k=k, nfeat=8)
    u = sc["u"] if pm == engine.PM_MSCKF_DELTAPOSE else sc["u"][:, [0, 1, 2, 10, 11, 12]]

    def run(Qx):
        f = engine.Msckf(B, nclones=k)
        f.set_state(sc["mu"], sc["P"])
        f.predict(pm, u, 0.01, Qx)
        return f.mu(), f.P(), f.status()

    a, b = run(sc["Q"]), run(_rep(sc["Q"]))
    for x, y in zip(a, b):
        np.testing.assert_array_equal(x, y)
    Q = _spd(np.random.default_rng(232), 12, np.abs(np.diag(sc["Q"])).mean())
    mu, P, st = run(Q)
    assert not st.any()
    ref = [slo.msckf_predict(pm, k, sc["mu"][i:i + 1], sc["P"][i:i + 1], u[i:i + 1], 0.01, Q[i]) for i in range(B)]
    mu_r = np.concatenate([r[0] for r in ref])
    P_r = parity.symmetrize_lower(np.concatenate([r[1] for r in ref]))
    parity.assert_parity(slo, synth.STATE_BLOCKS + [0, 1] * k, mu, P, mu_r, P_r)


# ---- isolation ----------------------------------------------------------------------------------------------------
def test_changing_one_instances_noise_changes_only_that_instance(slo):
    sc = synth.usckf_scenario(B, seed=241)
    Q, R = _usckf_noise(sc, 3, 242)
    a = _usckf(3, 9, "step", sc, Q, R)
    Q2, R2 = Q.copy(), R.copy()
    Q2[7] *= 3.0
    R2[7] = 0.5 * R[7] + 0.02 * np.eye(3)
    b = _usckf(3, 9, "step", sc, Q2, R2)
    others = np.arange(B) != 7
    for x, y in zip(a, b):
        np.testing.assert_array_equal(x[others], y[others])
    assert not np.array_equal(a[1][7], b[1][7])
    mu_r, P_r, st_r = _usckf_oracle(slo, 3, 9, "step", sc, Q2, R2, only=[7])
    parity.assert_parity(slo, AUG, b[0][7:8], b[1][7:8], mu_r, P_r, nfeat=12)
    # the same on a UKFoM batch
    su = synth.ukfom_scenario(B, seed=243)
    Qu, Ru = _ukf_noise(su, 9, 244)
    c = _ukf(9, engine.PM_UKFOM_IMU, "step", su, Qu, Ru)
    Qu2, Ru2 = Qu.copy(), Ru.copy()
    Qu2[7] *= 3.0
    Ru2[7] *= 5.0
    d = _ukf(9, engine.PM_UKFOM_IMU, "step", su, Qu2, Ru2)
    for x, y in zip(c, d):
        np.testing.assert_array_equal(x[others], y[others])
    mu_r, P_r, _ = _ukf_oracle(slo, 9, engine.PM_UKFOM_IMU, "step", su, Qu2, Ru2, only=[7])
    parity.assert_parity(slo, synth.LAYOUT_BLOCKS[9], d[0][7:8], d[1][7:8], mu_r, P_r)


# ---- gate ---------------------------------------------------------------------------------------------------------
def test_per_instance_r_decides_the_chi2_gate_per_instance(slo):
    """The same innovation passes the 5 % chi-square gate under a wide R and fails under a narrow one."""
    rng = np.random.default_rng(251)
    wide = rng.uniform(size=B) < 0.5
    sc = synth.usckf_scenario(B, seed=252)
    sc["z"] = sc["z"] + 0.3
    Q = _usckf_noise(sc, 3, 253)[0]
    R = np.where(wide[:, None, None], 1.0, 1e-4) * _rep(np.eye(3))
    for mode in ("update", "step"):
        mu, P, st = _usckf(3, 9, mode, sc, Q, R, gate=3)
        mu_r, P_r, st_r = _usckf_oracle(slo, 3, 9, mode, sc, Q, R, gate=3)
        np.testing.assert_array_equal(st, st_r)
        rej = (st & engine.ST_GATE_REJECT) != 0
        assert rej.any() and not rej.all()
        parity.assert_parity(slo, AUG, mu, P, mu_r, P_r, nfeat=12)
    su = synth.ukfom_scenario(B, seed=254)
    su["z"] = su["z"] + 0.3
    Qu = _ukf_noise(su, 9, 255)[0]
    Ru = np.where(wide[:, None, None], 1.0, 1e-6) * _rep(np.eye(3))
    for mode in ("update", "step"):
        mu, P, st = _ukf(9, engine.PM_UKFOM_IMU, mode, su, Qu, Ru, gate=3)
        mu_r, P_r, st_r = _ukf_oracle(slo, 9, engine.PM_UKFOM_IMU, mode, su, Qu, Ru, gate=3)
        np.testing.assert_array_equal(st, st_r)
        rej = (st & engine.ST_GATE_REJECT) != 0
        assert rej.any() and not rej.all()
        parity.assert_parity(slo, synth.LAYOUT_BLOCKS[9], mu, P, mu_r, P_r)


# ---- handle state -------------------------------------------------------------------------------------------------
def _raw_usckf_step(f, sc, Q, R):
    u, z, Qd, Rd = (engine.DeviceArray(np.ascontiguousarray(x)) for x in (sc["u"], sc["z"], Q, R))
    engine.check(engine.lib().slb_usckf_step(f.h, engine.PM_USCKF_TEST, engine.MM_USCKF_VO, u.ptr, sc["dt"], Qd.ptr, z.ptr,
                                             Rd.ptr, 0, engine._stream()))


def test_noise_layout_is_handle_state():
    sc = synth.usckf_scenario(B, seed=261)
    Q, R = _usckf_noise(sc, 3, 262)
    want = _usckf(3, 9, "step", sc, Q, R)
    shared = _usckf(3, 9, "step", sc, sc["Q"], sc["R"])
    f = engine.Usckf(B)
    f.set_state(sc["mu"], sc["P"])
    f.set_noise_layout(engine.NOISE_Q_PER_INSTANCE | engine.NOISE_R_PER_INSTANCE)
    _raw_usckf_step(f, sc, Q, R)                          # the raw ABI: the flags set earlier still hold
    for x, y in zip((f.mu(), f.P(), f.status()), want):
        np.testing.assert_array_equal(x, y)
    g = engine.Usckf(B)
    g.set_state(sc["mu"], sc["P"])
    g.set_noise_layout(engine.NOISE_R_PER_INSTANCE)
    g.set_noise_layout(0)                                 # back to the shared layout, bitwise
    _raw_usckf_step(g, sc, sc["Q"], sc["R"])
    for x, y in zip((g.mu(), g.P(), g.status()), shared):
        np.testing.assert_array_equal(x, y)


def test_noise_layout_refusals():
    L = engine.lib()
    u = engine.Ukf(64)
    s = engine.Usckf(64)
    m = engine.Msckf(64, nclones=2)
    for f in (u, s, m):
        for bad in (4, -1, 7):
            assert L.slb_set_noise_layout(f.h, bad) == -1
    assert L.slb_set_noise_layout(m.h, engine.NOISE_R_PER_INSTANCE) == -1
    assert b"MSCKF" in L.slb_last_error()
    assert L.slb_set_noise_layout(m.h, engine.NOISE_Q_PER_INSTANCE) == 0
    buf = np.zeros(64 * 200)
    p = buf.ctypes.data_as(C.c_void_p)
    dt = C.c_double(0.01)
    for flags in (engine.NOISE_Q_PER_INSTANCE, engine.NOISE_R_PER_INSTANCE):
        for f in (u, s):
            f.set_noise_layout(flags)
        calls = [
            lambda: L.slb_ukf_step_host(u.h, engine.PM_UKFOM_IMU, engine.MM_GPS_POS, p, dt, p, p, p, 0, None, None),
            lambda: L.slb_ukf_step_host_async(u.h, engine.PM_UKFOM_IMU, engine.MM_GPS_POS, p, dt, p, p, p, 0, None, None),
            lambda: L.slb_usckf_step_host(s.h, engine.PM_USCKF_TEST, engine.MM_USCKF_VO, p, dt, p, p, p, 0, None, None),
            lambda: L.slb_usckf_step_host_async(s.h, engine.PM_USCKF_TEST, engine.MM_USCKF_VO, p, dt, p, p, p, 0, None, None),
        ]
        if flags == engine.NOISE_Q_PER_INSTANCE:
            calls += [
                lambda: L.slb_msckf_step_host(m.h, engine.PM_MSCKF_DELTAPOSE, engine.MM_MSCKF_REPROJ, p, dt, p, p, 6, 4, p, p, 1,
                                              None, None),
                lambda: L.slb_msckf_step_host_async(m.h, engine.PM_MSCKF_DELTAPOSE, engine.MM_MSCKF_REPROJ, p, dt, p, p, 6, 4, p,
                                                    p, 1, None, None),
            ]
        for call in calls:
            assert call() == -1
            assert b"device-resident" in L.slb_last_error()
    assert not u.status().any() and not s.status().any() and not m.status().any()


def test_engine_refuses_malformed_noise_before_the_library():
    s = engine.Usckf(16)
    sc = synth.usckf_scenario(16, seed=271)
    s.set_state(sc["mu"], sc["P"])
    n0 = engine.launch_count()
    for Q in (np.eye(11), np.zeros((15, 12, 12)), np.zeros((16, 12, 13)), np.zeros(144)):
        with pytest.raises(ValueError):
            s.predict(engine.PM_USCKF_TEST, sc["u"], sc["dt"], Q)
    with pytest.raises(ValueError):
        s.update(engine.MM_USCKF_VO, sc["z"], np.zeros((16, 9, 9)))
    with pytest.raises(ValueError):
        s.set_measurement(engine.STATEK_L, np.zeros((16, 9)), np.eye(3))
    with pytest.raises(ValueError):
        s.step_host(engine.PM_USCKF_TEST, engine.MM_USCKF_VO, sc["u"], sc["dt"], _rep16(sc["Q"]), sc["z"], sc["R"],
                    mu_out=np.empty((16, 51)))
    u = engine.Ukf(16)
    with pytest.raises(ValueError):
        u.predict(engine.PM_UKFOM_IMU, np.zeros((16, 6)), 0.01, np.eye(6))
    m = engine.Msckf(16, nclones=2)
    with pytest.raises(ValueError):
        m.predict(engine.PM_MSCKF_DELTAPOSE, np.zeros((16, 13)), 0.01, np.zeros((16, 6, 6)))
    assert engine.launch_count() == n0 and s.noise == 0 and u.noise == 0 and m.noise == 0


def _rep16(M):
    return np.ascontiguousarray(np.broadcast_to(M, (16,) + M.shape))
