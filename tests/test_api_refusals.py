"""How the filter entry points refuse a call: the return code and the slb_last_error() text of every handle-taking
predict / update / step / step_host entry point, for a null handle (no GPU needed), a handle of another kind, missing
inputs, MSCKF measurement dimensions and models the update is not built for, and per-instance noise given to a host
step.  A refusal launches nothing.  Where a call breaks two rules, the message is the one of the rule checked first."""
import ctypes as C

import numpy as np
import pytest

from slam_localization_b200 import engine

INVALID = -1
UKF_KIND = b"slb_ukf_*: handle is not a UKF batch"
USCKF_KIND = b"slb_usckf_*: handle is not a USCKF batch"


def _call(fn, names, defaults):
    """lib().fn(h, *args): args by name from defaults, overridden by the keywords of the call."""
    def run(h, **kw):
        a = dict(defaults, **kw)
        return getattr(engine.lib(), fn)(h, *[a[n] for n in names])
    return run


def _device_calls(ptr):
    """name -> (kind the entry point serves, call(h, **overrides), its wrong-kind message).  Every pointer input is
    ptr; an override replaces any argument by name."""
    call, P = _call, engine
    ukf = dict(pm=P.PM_UKFOM_IMU, mm=P.MM_GPS_POS, dt=0.01, gate=0, stream=None)
    usc = dict(pm=P.PM_USCKF_TEST, mm=P.MM_USCKF_VO, dt=0.01, gate=0, stream=None)
    ms = dict(pm=P.PM_MSCKF_DELTAPOSE, mm=P.MM_MSCKF_REPROJ, dt=0.01, gate=1, m=4, mode=P.STATEK_I, stream=None)
    for d in (ukf, usc, ms):
        d.update(u=ptr, Q=ptr, z=ptr, R=ptr, params=ptr)
    pred, upd = ["pm", "u", "dt", "Q", "stream"], ["mm", "z", "R", "gate", "stream"]
    step = ["pm", "mm", "u", "dt", "Q", "z", "R", "gate", "stream"]
    msu = ["mm", "params", "m", "z", "R", "gate", "stream"]
    return {
        "slb_ukf_predict": (P.KIND_UKF, call("slb_ukf_predict", pred, ukf), UKF_KIND),
        "slb_ukf_update": (P.KIND_UKF, call("slb_ukf_update", upd, ukf), UKF_KIND),
        "slb_ukf_step": (P.KIND_UKF, call("slb_ukf_step", step, ukf), UKF_KIND),
        "slb_usckf_predict": (P.KIND_USCKF, call("slb_usckf_predict", pred, usc), USCKF_KIND),
        "slb_usckf_update": (P.KIND_USCKF, call("slb_usckf_update", upd, usc), USCKF_KIND),
        "slb_usckf_step": (P.KIND_USCKF, call("slb_usckf_step", step, usc), USCKF_KIND),
        "slb_usckf_clone": (P.KIND_USCKF, call("slb_usckf_clone", ["mode", "stream"], usc | {"mode": P.STATEK_I}),
                            b"slb_usckf_clone: handle is not a USCKF batch"),
        "slb_usckf_set_measurement": (P.KIND_USCKF, call("slb_usckf_set_measurement", ["mode", "z", "R", "stream"],
                                                         usc | {"mode": P.STATEK}),
                                      b"slb_usckf_set_measurement: handle is not a USCKF batch"),
        "slb_msckf_predict": (P.KIND_MSCKF, call("slb_msckf_predict", pred, ms),
                              b"slb_msckf_predict: handle is not an MSCKF batch"),
        "slb_msckf_update": (P.KIND_MSCKF, call("slb_msckf_update", msu, ms),
                             b"slb_msckf_update: handle is not an MSCKF batch"),
        "slb_msckf_update_ekf": (P.KIND_MSCKF, call("slb_msckf_update_ekf", msu, ms),
                                 b"slb_msckf_update_ekf: handle is not an MSCKF batch"),
    }


def _host_steps(ptr):
    """The six *_step_host[_async] entry points, as _device_calls."""
    call, P = _call, engine
    common = dict(dt=0.01, gate=0, mu_out=None, stream=None, u=ptr, Q=ptr, z=ptr, R=ptr, params=ptr)
    ukf = dict(common, pm=P.PM_UKFOM_IMU, mm=P.MM_GPS_POS)
    usc = dict(common, pm=P.PM_USCKF_TEST, mm=P.MM_USCKF_VO)
    ms = dict(common, pm=P.PM_MSCKF_DELTAPOSE, mm=P.MM_MSCKF_REPROJ, nparams=12, m=4, gate=1)
    sh = ["pm", "mm", "u", "dt", "Q", "z", "R", "gate", "mu_out", "stream"]
    msh = ["pm", "mm", "u", "dt", "Q", "params", "nparams", "m", "z", "R", "gate", "mu_out", "stream"]
    out = {}
    for sfx in ("", "_async"):
        out["slb_ukf_step_host" + sfx] = (P.KIND_UKF, call("slb_ukf_step_host" + sfx, sh, ukf),
                                          b"slb_ukf_step_host: handle is not a UKF batch")
        out["slb_usckf_step_host" + sfx] = (P.KIND_USCKF, call("slb_usckf_step_host" + sfx, sh, usc),
                                            b"slb_usckf_step_host: handle is not a USCKF batch")
        out["slb_msckf_step_host" + sfx] = (P.KIND_MSCKF, call("slb_msckf_step_host" + sfx, msh, ms),
                                            b"slb_msckf_step_host: handle is not an MSCKF batch")
    return out


def _refused(call, h, msg, **kw):
    n0 = engine.launch_count()
    rc = call(h, **kw)
    assert (rc, engine.lib().slb_last_error()) == (INVALID, msg)
    assert engine.launch_count() == n0


_NULLS = dict(u=None, Q=None, z=None, R=None, params=None, m=0, nparams=0, mm=0)


@pytest.mark.parametrize("name", sorted(_device_calls(None)))
def test_device_call_refuses_a_null_handle(name):
    # every other input is missing too: the handle is checked first
    _, call, msg = _device_calls(None)[name]
    _refused(call, None, msg, **_NULLS)


@pytest.mark.parametrize("name", sorted(_host_steps(None)))
def test_host_step_refuses_a_null_handle(name):
    _, call, msg = _host_steps(None)[name]
    _refused(call, None, msg, **_NULLS)


def test_entry_points_without_a_device_name_themselves():
    """Without a CUDA device every entry point that would start device work answers SLB_ERR_NO_DEVICE in its own words."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    L, P = engine.lib(), engine
    buf = np.zeros(4096)
    p = buf.ctypes.data_as(C.c_void_p)
    acc = (C.c_int32 * 4)()
    cfg = P.SlbConfig()
    cfg.kind, cfg.layout, cfg.batch = P.KIND_UKF, P.LAYOUT_MTK9, 8
    full = b": no CUDA device (this engine has no CPU fallback)"
    cases = [
        (lambda: L.slb_create(C.byref(cfg), C.byref(C.c_void_p())), b"slb_create" + full),
        (lambda: L.slb_datamodel_fuse_host(6, 1, p, p, p, p, p, p), b"slb_datamodel_fuse_host: no CUDA device (no CPU fallback)"),
        (lambda: L.slb_dev_alloc(C.c_size_t(8), C.byref(C.c_void_p())), b"slb_dev_alloc" + full),
        (lambda: L.slb_bench_fp64_peak(C.byref(C.c_double())), b"slb_bench_fp64_peak: no CUDA device"),
        (lambda: L.slb_ekf_predict(1, p, p, p, p, None), b"slb_ekf_predict" + full),
        (lambda: L.slb_ekf_update(1, 3, p, p, p, p, p, 0, p, acc, None), b"slb_ekf_update" + full),
        (lambda: L.slb_ekf_single_update(1, 3, p, p, p, p, p, p, 0, acc, None), b"slb_ekf_single_update" + full),
        (lambda: L.slb_ekf_clone(1, p, p, p, None), b"slb_ekf_clone" + full),
        (lambda: L.slb_datamodel_safe_fuse(1, p, p, p, p, p, p, None), b"slb_datamodel_safe_fuse" + full),
        (lambda: L.slb_transform_compose(1, p, p, p, p, p, p, None), b"slb_transform_compose" + full),
        (lambda: L.slb_deadreckon_update_pose(1, C.c_double(0.01), p, p, p, p, p, p, p, p, p, None),
         b"slb_deadreckon_update_pose" + full),
    ]
    for call, msg in cases:
        assert (call(), L.slb_last_error()) == (-2, msg)


# ---- GPU: real handles ---------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def batches():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    b = {engine.KIND_UKF: engine.Ukf(64, layout=engine.LAYOUT_MTK9),
         engine.KIND_USCKF: engine.Usckf(64, nk=3, nl=9),
         engine.KIND_MSCKF: engine.Msckf(64, nclones=2)}
    yield b
    for x in b.values():
        x.close()


@pytest.fixture(scope="module")
def dev_ptr(batches):
    """Every input of a device call points into one zeroed device buffer (a refused call reads none of it)."""
    buf = engine.DeviceArray(np.zeros(1 << 16))
    yield buf.ptr
    del buf


@pytest.fixture(scope="module")
def host_ptr():
    buf = np.zeros(1 << 16)
    yield buf.ctypes.data_as(C.c_void_p)
    del buf


@pytest.mark.gpu
@pytest.mark.parametrize("kind", [engine.KIND_UKF, engine.KIND_USCKF, engine.KIND_MSCKF])
def test_device_calls_refuse_a_handle_of_another_kind(batches, dev_ptr, kind):
    for name, (serves, call, msg) in _device_calls(dev_ptr).items():
        if serves != kind:
            _refused(call, batches[kind].h, msg)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", [engine.KIND_UKF, engine.KIND_USCKF, engine.KIND_MSCKF])
def test_host_steps_refuse_a_handle_of_another_kind(batches, host_ptr, kind):
    for name, (serves, call, msg) in _host_steps(host_ptr).items():
        if serves != kind:
            _refused(call, batches[kind].h, msg)


@pytest.mark.gpu
@pytest.mark.parametrize("f", ["ukf", "usckf"])
def test_ukf_usckf_device_calls_refuse_missing_inputs(batches, dev_ptr, f):
    kind = engine.KIND_UKF if f == "ukf" else engine.KIND_USCKF
    calls, h = _device_calls(dev_ptr), batches[kind].h
    no_pred = ("slb_%s_predict: u and Q are required" % f).encode()
    no_upd = ("slb_%s_update: z and R are required" % f).encode()
    for x in ("u", "Q"):
        _refused(calls["slb_%s_predict" % f][1], h, no_pred, **{x: None})
        _refused(calls["slb_%s_step" % f][1], h, no_pred, **{x: None})
    for x in ("z", "R"):
        _refused(calls["slb_%s_update" % f][1], h, no_upd, **{x: None})
        _refused(calls["slb_%s_step" % f][1], h, no_upd, **{x: None})
    _refused(calls["slb_%s_step" % f][1], h, no_pred, u=None, z=None)   # predict inputs are checked first


@pytest.mark.gpu
def test_usckf_set_measurement_refuses_missing_inputs(batches, dev_ptr):
    call, h = _device_calls(dev_ptr)["slb_usckf_set_measurement"][1], batches[engine.KIND_USCKF].h
    for x in ("z", "R"):
        _refused(call, h, b"slb_usckf_set_measurement: z and R are required", **{x: None})


@pytest.mark.gpu
def test_device_calls_refuse_models_they_are_not_built_for(batches, dev_ptr):
    calls, P = _device_calls(dev_ptr), engine
    h = batches[P.KIND_UKF].h
    for name in ("slb_ukf_update", "slb_ukf_step"):
        _refused(calls[name][1], h, b"ukf: unsupported measurement model", mm=P.MM_USCKF_VO)
    for name in ("slb_ukf_predict", "slb_ukf_step"):
        _refused(calls[name][1], h, b"ukf: unsupported layout / process model combination", pm=P.PM_POSE6_ODOM)
    h = batches[P.KIND_USCKF].h
    for name in ("slb_usckf_update", "slb_usckf_step"):
        _refused(calls[name][1], h, b"usckf: unsupported measurement model", mm=P.MM_GPS_POS)
    for name in ("slb_usckf_predict", "slb_usckf_step"):
        _refused(calls[name][1], h, b"usckf: unsupported process model", pm=P.PM_UKFOM_IMU)
    h = batches[P.KIND_MSCKF].h
    _refused(calls["slb_msckf_predict"][1], h, b"msckf: unsupported process model", pm=P.PM_UKFOM_IMU)
    for name in ("slb_msckf_update", "slb_msckf_update_ekf"):
        _refused(calls[name][1], h, b"msckf: unsupported measurement model", mm=P.MM_GPS_POS)


@pytest.mark.gpu
def test_msckf_device_calls_refuse_missing_inputs_and_bad_m(batches, dev_ptr):
    calls, h = _device_calls(dev_ptr), batches[engine.KIND_MSCKF].h
    for x in ("u", "Q"):
        _refused(calls["slb_msckf_predict"][1], h, b"slb_msckf_predict: u and Q are required", **{x: None})
    for name in ("slb_msckf_update", "slb_msckf_update_ekf"):
        bad = (name + ": bad arguments").encode()
        for kw in (dict(params=None), dict(z=None), dict(R=None), dict(m=0), dict(m=-2), dict(m=3), dict(m=5),
                   dict(m=3, mm=engine.MM_GPS_POS)):   # an odd m is refused before the model is looked at
            _refused(calls[name][1], h, bad, **kw)


@pytest.mark.gpu
def test_host_steps_refuse_missing_inputs(batches, host_ptr):
    steps, P = _host_steps(host_ptr), engine
    for sfx in ("", "_async"):
        for f, kind in (("ukf", P.KIND_UKF), ("usckf", P.KIND_USCKF)):
            call, h = steps["slb_%s_step_host%s" % (f, sfx)][1], batches[kind].h
            for x in ("u", "Q", "z", "R"):
                _refused(call, h, b"slb_*_step_host: null argument", **{x: None})
        # the UKF host step checks its measurement model before its inputs
        _refused(steps["slb_ukf_step_host" + sfx][1], batches[P.KIND_UKF].h, b"ukf: unsupported measurement model",
                 u=None, mm=P.MM_USCKF_VO)
        call, h = steps["slb_msckf_step_host" + sfx][1], batches[P.KIND_MSCKF].h
        null = b"slb_msckf_step_host: null argument"
        for kw in (dict(u=None), dict(Q=None), dict(params=None), dict(z=None), dict(R=None), dict(m=0), dict(nparams=0),
                   dict(u=None, m=3)):
            _refused(call, h, null, **kw)
        for kw in (dict(m=3), dict(mm=P.MM_GPS_POS)):
            _refused(call, h, b"slb_msckf_step_host: bad measurement model / m", **kw)


@pytest.mark.gpu
@pytest.mark.parametrize("kind,f", [(engine.KIND_UKF, "ukf"), (engine.KIND_USCKF, "usckf"), (engine.KIND_MSCKF, "msckf")])
def test_host_steps_refuse_per_instance_noise(batches, host_ptr, kind, f):
    b = batches[kind]
    b.set_noise_layout(engine.NOISE_Q_PER_INSTANCE)
    try:
        msg = ("slb_%s_step_host: per-instance noise (slb_set_noise_layout) is device-resident only" % f).encode()
        for sfx in ("", "_async"):
            call = _host_steps(host_ptr)["slb_%s_step_host%s" % (f, sfx)][1]
            _refused(call, b.h, msg)
            _refused(call, b.h, msg, **_NULLS)   # checked before the model and the inputs
    finally:
        b.set_noise_layout(0)
