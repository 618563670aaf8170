"""Filter consistency on the GPU: the NIS every UKFoM / USCKF update captures (slb_set_nis_capture) and the NEES of
slb_consistency_stats against a per-instance truth.

The captured m2 is compared with a numpy restatement of the update's distance (tests/consistency_ref.py), evaluated on
the prior the update saw: the uploaded state for update calls, the CPU oracle's prediction for step calls."""
import ctypes as C
import threading

import numpy as np
import pytest

import consistency_ref as cref
from slam_localization_b200 import engine, fleet, synth

pytestmark = pytest.mark.gpu
B = 203                  # ragged against the 8-instance UKF warps and the 4- / 6-warp USCKF CTAs
ALL_SHAPES = [(3, 0), (3, 3), (3, 6), (3, 9), (6, 0), (6, 3), (6, 6), (9, 0), (9, 3)]
UKF_CASES = [(9, engine.PM_UKFOM_IMU), (6, engine.PM_POSE6_ODOM)]
AUG = synth.STATE_BLOCKS * 3
RTOL = 1e-9


def _nis_close(got, want):
    np.testing.assert_allclose(got, want, rtol=RTOL, atol=0)


# ---- runners ------------------------------------------------------------------------------------------------------
def _ukf(layout, pm, mode, sc, Q, R, gate=0, capture=True, P=None):
    f = engine.Ukf(len(sc["mu"]), layout=layout)
    f.set_state(sc["mu"], sc["P"] if P is None else P)
    if capture:
        f.set_nis_capture(True)
    if mode == "predict":
        f.predict(pm, sc["u"], sc["dt"], Q)
    elif mode == "update":
        f.update(engine.MM_GPS_POS, sc["z"], R, gate_dof=gate)
    else:
        f.step(pm, engine.MM_GPS_POS, sc["u"], sc["dt"], Q, sc["z"], R, gate_dof=gate)
    return f


def _usckf(nk, nl, mode, sc, Q, R, gate=0, capture=True, P=None):
    f = engine.Usckf(len(sc["mu"]), nk=nk, nl=nl)
    f.set_state(sc["mu"], sc["P"] if P is None else P)
    if capture:
        f.set_nis_capture(True)
    if mode == "predict":
        f.predict(engine.PM_USCKF_TEST, sc["u"], sc["dt"], Q)
    elif mode == "update":
        f.update(engine.MM_USCKF_VO, sc["z"], R, gate_dof=gate)
    else:
        f.step(engine.PM_USCKF_TEST, engine.MM_USCKF_VO, sc["u"], sc["dt"], Q, sc["z"], R, gate_dof=gate)
    return f


def _noise(M, i):
    return M[i] if M.ndim == 3 else M


def _ukf_ref(slo, layout, pm, mode, sc, Q, R):
    mu, P = sc["mu"], sc["P"]
    out = np.empty(len(mu))
    for i in range(len(mu)):
        m, p = mu[i], P[i]
        if mode == "step":
            mo, po, _, _ = slo.ukf_step(layout, pm, slo.MM_GPS_POS, mu[i:i + 1], P[i:i + 1], sc["u"][i:i + 1], sc["dt"],
                                        _noise(Q, i), None, None, predict=True, update=False)
            m, p = mo[0], po[0]
        out[i] = cref.ukf_m2(m, p, sc["z"][i], _noise(R, i))
    return out


def _usckf_ref(slo, nk, nl, mode, sc, Q, R):
    mu, P = sc["mu"], sc["P"]
    out = np.empty(len(mu))
    for i in range(len(mu)):
        m, p = mu[i], P[i]
        if mode == "step":
            mo, po, _, _ = slo.usckf_step(slo.PM_USCKF_TEST, slo.MM_USCKF_VO, nk, nl, mu[i:i + 1], P[i:i + 1], sc["u"][i:i + 1],
                                          sc["dt"], _noise(Q, i), None, None, predict=True, update=False)
            m, p = mo[0], po[0]
        out[i] = cref.usckf_m2(nk, m, p, sc["z"][i], _noise(R, i))
    return out


# ---- 1. NIS matches the reference distance ------------------------------------------------------------------------
@pytest.mark.parametrize("layout,pm", UKF_CASES)
@pytest.mark.parametrize("mode", ["update", "step"])
def test_ukf_nis_matches_reference(slo, layout, pm, mode):
    sc = synth.ukfom_scenario(B, seed=601, layout=layout)
    f = _ukf(layout, pm, mode, sc, sc["Q"], sc["R"])
    assert not f.status().any()
    _nis_close(f.nis(), _ukf_ref(slo, layout, pm, mode, sc, sc["Q"], sc["R"]))


@pytest.mark.parametrize("nk,nl", ALL_SHAPES)
@pytest.mark.parametrize("mode", ["update", "step"])
def test_usckf_nis_matches_reference(slo, nk, nl, mode):
    sc = synth.usckf_scenario(B, seed=611, nk=nk, nl=nl)
    f = _usckf(nk, nl, mode, sc, sc["Q"], sc["R"])
    assert not f.status().any()
    _nis_close(f.nis(), _usckf_ref(slo, nk, nl, mode, sc, sc["Q"], sc["R"]))


def test_nis_with_per_instance_noise(slo):
    rng = np.random.default_rng(621)
    su = synth.ukfom_scenario(B, seed=622)
    Qu = synth.random_spd(rng, B, 9, 1e-5, 10.0)
    Ru = synth.random_spd(rng, B, 3, 1e-4, 10.0) * 10.0 ** rng.uniform(-1, 1, size=(B, 1, 1))
    for mode in ("update", "step"):
        f = _ukf(9, engine.PM_UKFOM_IMU, mode, su, Qu, Ru)
        _nis_close(f.nis(), _ukf_ref(slo, 9, engine.PM_UKFOM_IMU, mode, su, Qu, Ru))
    ss = synth.usckf_scenario(B, seed=623, nk=6, nl=3)
    Qs = synth.random_spd(rng, B, 12, 1e-3, 10.0)
    Rs = synth.random_spd(rng, B, 6, 1e-2, 10.0) * 10.0 ** rng.uniform(-1, 1, size=(B, 1, 1))
    for mode in ("update", "step"):
        f = _usckf(6, 3, mode, ss, Qs, Rs)
        _nis_close(f.nis(), _usckf_ref(slo, 6, 3, mode, ss, Qs, Rs))


# ---- 2. the gate decides on exactly the captured value ------------------------------------------------------------
def test_gate_agrees_with_nis_exactly():
    su = synth.ukfom_scenario(B, seed=631)
    su["z"] = su["z"] + 0.03
    ss = synth.usckf_scenario(B, seed=632)
    ss["z"] = ss["z"] + 0.15
    for mode in ("update", "step"):
        for f in (_ukf(9, engine.PM_UKFOM_IMU, mode, su, su["Q"], su["R"], gate=3),
                  _usckf(3, 9, mode, ss, ss["Q"], ss["R"], gate=3)):
            rej = (f.status() & engine.ST_GATE_REJECT) != 0
            assert rej.any() and not rej.all()
            np.testing.assert_array_equal(rej, f.nis() >= cref.CHI2_5[3])


# ---- 3. failed updates give NaN, the others are untouched ---------------------------------------------------------
def test_failed_updates_give_nan():
    bad = np.zeros(B, bool)
    bad[[0, 5, 77, 202]] = True
    su = synth.ukfom_scenario(B, seed=641)
    ss = synth.usckf_scenario(B, seed=642)
    for sc, run, args in ((su, _ukf, (9, engine.PM_UKFOM_IMU)), (ss, _usckf, (3, 9))):
        P = sc["P"].copy()
        P[bad] = -P[bad]
        for mode in ("update", "step"):
            good = run(*args, mode, sc, sc["Q"], sc["R"]).nis()
            f = run(*args, mode, sc, sc["Q"], sc["R"], P=P)
            nis, st = f.nis(), f.status()
            assert np.isnan(nis[bad]).all() and ((st[bad] & engine.ST_CHOL_FAIL) != 0).all()
            np.testing.assert_array_equal(nis[~bad], good[~bad])
            assert not st[~bad].any()


# ---- 4. capture changes no result; host steps and the graph key --------------------------------------------------
def _state(f):
    return f.mu(), f.P(), f.status()


def _assert_same(a, b):
    for x, y in zip(a, b):
        np.testing.assert_array_equal(x, y)


@pytest.mark.parametrize("mode", ["predict", "update", "step"])
def test_capture_changes_no_result(mode):
    for layout, pm in UKF_CASES:
        sc = synth.ukfom_scenario(B, seed=651, layout=layout)
        sc["z"] = sc["z"] + 0.02
        for gate in (0, 3):
            _assert_same(_state(_ukf(layout, pm, mode, sc, sc["Q"], sc["R"], gate, True)),
                         _state(_ukf(layout, pm, mode, sc, sc["Q"], sc["R"], gate, False)))
    for nk, nl in ALL_SHAPES:
        sc = synth.usckf_scenario(B, seed=652, nk=nk, nl=nl)
        _assert_same(_state(_usckf(nk, nl, mode, sc, sc["Q"], sc["R"], 0, True)),
                     _state(_usckf(nk, nl, mode, sc, sc["Q"], sc["R"], 0, False)))
    if mode == "predict":   # predict-only calls leave the array alone
        f = _usckf(3, 9, "predict", sc, sc["Q"], sc["R"])
        assert np.isnan(f.nis()).all()


def test_host_steps_capture_what_the_device_step_captures():
    import torch
    cases = [(engine.Ukf, synth.ukfom_scenario(B, seed=661), engine.PM_UKFOM_IMU, engine.MM_GPS_POS),
             (engine.Usckf, synth.usckf_scenario(B, seed=662), engine.PM_USCKF_TEST, engine.MM_USCKF_VO)]
    for cls, sc, pm, mm in cases:
        dev = cls(B)
        dev.set_state(sc["mu"], sc["P"])
        dev.set_nis_capture(True)
        for _ in range(2):
            dev.step(pm, mm, sc["u"], sc["dt"], sc["Q"], sc["z"], sc["R"])
        for pin in (False, True):   # pageable buffers: the copy pipeline; page-locked ones: the zero-copy kernels
            h = cls(B)
            h.set_state(sc["mu"], sc["P"])
            h.set_nis_capture(True)
            u, Q, z, R = [torch.from_numpy(np.ascontiguousarray(a)).pin_memory() if pin else a
                          for a in (sc["u"], sc["Q"], sc["z"], sc["R"])]
            h.step_host(pm, mm, u, sc["dt"], Q, z, R)
            h.step_host(pm, mm, u, sc["dt"], Q, z, R, wait=False)
            h.wait()
            np.testing.assert_array_equal(h.nis(), dev.nis())
            _assert_same(_state(h), _state(dev))


_GRAPH_SCRIPT = r"""
import sys
import numpy as np, torch
sys.path[:0] = [sys.argv[1], sys.argv[1] + "/tests"]
from slam_localization_b200 import engine, synth
B = 203
sc = synth.usckf_scenario(B, seed=671)
u, Q, z, R = [torch.from_numpy(np.ascontiguousarray(a)).pin_memory() for a in (sc["u"], sc["Q"], sc["z"], sc["R"])]
pm, mm = engine.PM_USCKF_TEST, engine.MM_USCKF_VO
ref = engine.Usckf(B)
ref.set_state(sc["mu"], sc["P"])
ref.set_nis_capture(True)
h = engine.Usckf(B)
h.set_state(sc["mu"], sc["P"])
counts = []
for on in (True, False, True, True):
    h.set_nis_capture(on)
    n0 = engine.launch_count()
    h.step_host(pm, mm, u, sc["dt"], Q, z, R)
    counts.append(engine.launch_count() - n0)
    ref.step(pm, mm, sc["u"], sc["dt"], sc["Q"], sc["z"], sc["R"])
    if on:
        assert np.array_equal(h.nis(), ref.nis()), "a replayed graph missed the NIS array"
assert len(set(counts)) == 1, counts
for x, y in zip((h.mu(), h.P(), h.status()), (ref.mu(), ref.P(), ref.status())):
    assert np.array_equal(x, y)
print("OK", counts)
"""


def test_toggling_capture_recaptures_the_host_step_graph(tmp_path):
    """With SLB_ZERO_COPY=0 and page-locked buffers the host step is a captured CUDA graph, replayed while its key holds.
    The NIS array is part of the key: after capture is turned off and on again the replay writes the new array."""
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, SLB_ZERO_COPY="0")
    p = subprocess.run([sys.executable, "-c", _GRAPH_SCRIPT, root], capture_output=True, text=True, env=env, timeout=600)
    assert p.returncode == 0 and "OK" in p.stdout, p.stdout + p.stderr


# ---- 5. NEES known answer -----------------------------------------------------------------------------------------
def _known_truth(rng, blocks, nfeat, mu, P):
    w = rng.normal(size=(len(mu), P.shape[1]))
    return cref.boxplus(blocks, nfeat, mu, np.einsum("bij,bj->bi", np.linalg.cholesky(P), w)), w


def _nees_cases(f, blocks, nfeat, mu, P, ranges, seed):
    rng = np.random.default_rng(seed)
    truth, w = _known_truth(rng, blocks, nfeat, mu, P)
    out, ne = f.consistency_stats(truth, nees=True)
    np.testing.assert_allclose(ne, (w * w).sum(axis=1), rtol=RTOL)
    assert out[0] == len(mu)
    for t0, n in ranges:
        _, ne = f.consistency_stats(truth, t0=t0, n=n, nees=True)
        np.testing.assert_allclose(ne, cref.nees(blocks, nfeat, truth, mu, P, t0, n), rtol=RTOL)


@pytest.mark.parametrize("nk,nl", [(3, 9), (6, 0)])
def test_nees_known_answer_usckf(nk, nl):
    sc = synth.usckf_scenario(B, seed=681, nk=nk, nl=nl)
    f = engine.Usckf(B, nk=nk, nl=nl)
    f.set_state(sc["mu"], sc["P"])
    N = 36 + nk + nl
    _nees_cases(f, AUG, nk + nl, sc["mu"], sc["P"], [(24, 12), (27, 3), (36, nk + nl)], 682)
    assert N == f.N


def test_nees_known_answer_ukfom():
    sc = synth.ukfom_scenario(B, seed=691)
    f = engine.Ukf(B)
    f.set_state(sc["mu"], sc["P"])
    _nees_cases(f, [0, 1, 0], 0, sc["mu"], sc["P"], [(3, 3)], 692)


def test_nees_known_answer_msckf():
    sc = synth.msckf_scenario(B, seed=701, k=10, nfeat=4)
    f = engine.Msckf(B, nclones=10)
    f.set_state(sc["mu"], sc["P"])
    _nees_cases(f, synth.STATE_BLOCKS + [0, 1] * 10, 0, sc["mu"], sc["P"], [(18, 6)], 702)


# ---- 6. invalid instances drop out; range refusals ----------------------------------------------------------------
def test_invalid_instances_are_excluded_and_ranges_refused():
    sc = synth.usckf_scenario(B, seed=711)
    P = sc["P"].copy()
    bad = np.zeros(B, bool)
    bad[[3, 100]] = True
    P[bad, 24:36, 24:36] *= -1.0
    f = engine.Usckf(B)
    f.set_state(sc["mu"], P)
    truth = _known_truth(np.random.default_rng(712), AUG, 12, sc["mu"], sc["P"])[0]
    truth[50, 26] = np.nan                   # statek_i's position: inside [24, 36)
    out, ne = f.consistency_stats(truth, t0=24, n=12, nees=True)
    bad[50] = True
    assert np.isnan(ne[bad]).all() and np.isfinite(ne[~bad]).all()
    assert out[0] == (~bad).sum()
    L = engine.lib()
    o = engine.DeviceArray(shape=(6,))
    t = engine.dev(truth)
    n0 = engine.launch_count()
    for t0, n in ((1, 12), (24, 11), (0, 0), (-3, 6), (45, 6), (0, 49)):
        assert L.slb_consistency_stats(f.h, t.ptr, t0, n, None, o.ptr, None) == -1
    assert L.slb_consistency_stats(f.h, None, 0, 6, None, o.ptr, None) == -1
    assert L.slb_consistency_stats(f.h, t.ptr, 37, 2, None, o.ptr, None) == 0    # inside the features: any cut
    assert engine.launch_count() == n0 + 1
    assert not f.status().any()
    # NIS field refusals
    assert L.slb_device_ptr(f.h, engine.FIELD_NIS, C.byref(C.c_void_p())) == -1
    buf = np.zeros(B)
    assert L.slb_download(f.h, engine.FIELD_NIS, engine._hp(buf), B, None) == -1
    f.set_nis_capture(True)
    assert L.slb_upload(f.h, engine.FIELD_NIS, engine._hp(buf), B, None) == -1
    assert L.slb_device_ptr(f.h, engine.FIELD_NIS, C.byref(C.c_void_p())) == 0
    m = engine.Msckf(8, nclones=1)
    assert L.slb_set_nis_capture(m.h, 1) == -1 and b"MSCKF" in L.slb_last_error()


# ---- 7. sums and independence -------------------------------------------------------------------------------------
def test_sums_and_independence():
    sc = synth.usckf_scenario(B, seed=721)
    truth = _known_truth(np.random.default_rng(722), AUG, 12, sc["mu"], sc["P"])[0]
    f = _usckf(3, 9, "update", sc, sc["Q"], sc["R"])
    out, ne = f.consistency_stats(truth, nees=True)
    nis = f.nis()
    want = [len(ne), ne.sum(), (ne * ne).sum(), len(nis), nis.sum(), (nis * nis).sum()]
    np.testing.assert_allclose(out, want, rtol=1e-12)
    np.testing.assert_allclose(f.consistency_stats(), [0, 0, 0] + want[3:], rtol=1e-12)
    for i in (0, 101, 202):
        one = {k: (v[i:i + 1] if isinstance(v, np.ndarray) and v.shape[:1] == (B,) else v) for k, v in sc.items()}
        g = _usckf(3, 9, "update", one, sc["Q"], sc["R"])
        _, ne1 = g.consistency_stats(truth[i:i + 1], nees=True)
        assert ne1[0] == ne[i] and g.nis()[0] == nis[i]


# ---- 8. statistical check -----------------------------------------------------------------------------------------
def test_anees_inside_the_99_percent_interval():
    Bs = 65536
    sc = synth.ukfom_scenario(Bs, seed=731)
    f = engine.Ukf(Bs)
    f.set_state(sc["mu"], sc["P"])
    truth = _known_truth(np.random.default_rng(732), [0, 1, 0], 0, sc["mu"], sc["P"])[0]
    r = fleet.consistency(f.consistency_stats(truth), nees_dof=9, nis_dof=3, p=0.99)
    lo, hi = r["anees_interval"]
    assert r["anees_count"] == Bs and lo < r["anees"] < hi, r


# ---- 9. gather over NCCL ------------------------------------------------------------------------------------------
def test_gather_consistency_one_rank_equals_local():
    sc = synth.usckf_scenario(B, seed=741)
    truth = _known_truth(np.random.default_rng(742), AUG, 12, sc["mu"], sc["P"])[0]
    f = _usckf(3, 9, "update", sc, sc["Q"], sc["R"])
    try:
        comm = engine.NcclComm(0, 1, lambda raw: raw)
    except engine.SlbError as e:
        pytest.skip("NCCL unavailable: %s" % e)
    try:
        # (the sums are FP64 atomics: two calls agree to rounding, not bit for bit)
        np.testing.assert_allclose(f.gather_consistency(comm, truth, 24, 12), f.consistency_stats(truth, 24, 12), rtol=1e-12)
        np.testing.assert_allclose(f.gather_consistency(None, truth), f.consistency_stats(truth), rtol=1e-12)
    finally:
        comm.close()


def test_gather_consistency_two_devices():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("one device")
    sc = synth.usckf_scenario(2 * B, seed=751)
    truth = _known_truth(np.random.default_rng(752), AUG, 12, sc["mu"], sc["P"])[0]
    shards, local = [], []
    for d in range(2):
        with torch.cuda.device(d):
            s = {k: (v[d * B:(d + 1) * B] if isinstance(v, np.ndarray) and v.shape[:1] == (2 * B,) else v) for k, v in sc.items()}
            f = _usckf(3, 9, "update", s, sc["Q"], sc["R"])
            shards.append((f, truth[d * B:(d + 1) * B]))
            local.append(f.consistency_stats(shards[-1][1]))
    ident = (C.c_ubyte * 128)()
    engine.check(engine.lib().slb_nccl_unique_id(ident))
    comms, res = [None, None], [None, None]

    def go(r):   # one thread per rank: ncclCommInitRank blocks until every rank has joined
        with torch.cuda.device(r):
            comms[r] = engine.NcclComm(r, 2, lambda raw: bytes(ident), device=r)
            res[r] = shards[r][0].gather_consistency(comms[r], shards[r][1])
    ths = [threading.Thread(target=go, args=(r,)) for r in range(2)]
    for t in ths:
        t.start()
    for t in ths:
        t.join()
    for r in range(2):
        np.testing.assert_allclose(res[r], local[0] + local[1], rtol=1e-12)
        comms[r].close()
