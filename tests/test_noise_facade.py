"""Per-instance noise through the host C++ facade: tests/facade_noise_test.cpp runs one USCKF predict + update with a Q
and an R per instance, and its results must be the Python engine's, bit for bit.  Without a GPU the binary must refuse
to compute."""
import os
import subprocess

import numpy as np
import pytest

from slam_localization_b200 import build as slb_build
from slam_localization_b200 import engine, synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EXE = os.path.join(ROOT, "tests", "_build", "facade_noise_test")


def _build():
    slb_build.build()
    os.makedirs(os.path.dirname(EXE), exist_ok=True)
    src = os.path.join(ROOT, "tests", "facade_noise_test.cpp")
    hdr = os.path.join(ROOT, "slam-localization_b200", "facade", "localization_b200.hpp")
    if not os.path.exists(EXE) or os.path.getmtime(EXE) < max(os.path.getmtime(src), os.path.getmtime(hdr)):
        csrc = os.path.join(ROOT, "slam-localization_b200", "csrc")
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-o", EXE, src, "-L" + csrc, "-lslb", "-Wl,-rpath," + csrc,
                               "-L/usr/local/cuda/lib64", "-Wl,-rpath,/usr/local/cuda/lib64"])
    return EXE


def _scenario(B, nk=3, nl=9, seed=301):
    sc = synth.usckf_scenario(B, seed=seed, nk=nk, nl=nl)
    rng = np.random.default_rng(seed + 1)
    sc["Qi"] = synth.random_spd(rng, B, 12, 1.0, 10.0) * (1e-4 * 10.0 ** rng.uniform(-1, 1, size=(B, 1, 1)))
    sc["Ri"] = synth.random_spd(rng, B, nk, 1.0, 10.0) * (1e-2 * 10.0 ** rng.uniform(-1, 1, size=(B, 1, 1)))
    return sc


def _run(tmp_path, sc, B, nk=3, nl=9):
    fin, fout = str(tmp_path / "in.bin"), str(tmp_path / "out.bin")
    parts = [np.array([B, nk, nl, sc["dt"]], float), sc["mu"], sc["P"], sc["u"], sc["Qi"], sc["z"], sc["Ri"]]
    np.concatenate([np.ravel(p) for p in parts]).astype(np.float64).tofile(fin)
    p = subprocess.run([_build(), fin, fout], capture_output=True, text=True)
    return p, fout


def test_facade_noise_driver_compiles_and_refuses_without_gpu(tmp_path):
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present: covered by the GPU test below")
    p, _ = _run(tmp_path, _scenario(4), 4)
    assert p.returncode == 3 and "NO_DEVICE" in p.stdout


@pytest.mark.gpu
def test_facade_per_instance_noise_equals_engine(tmp_path):
    B, nk, nl = 37, 3, 9
    sc = _scenario(B)
    p, fout = _run(tmp_path, sc, B)
    assert p.returncode == 0 and "BADLEN" in p.stdout and "OK" in p.stdout, p.stdout + p.stderr
    N, QD = 36 + nk + nl, 39 + nk + nl
    out = np.fromfile(fout, dtype=np.float64)
    mu, P, st = out[:B * QD].reshape(B, QD), out[B * QD:B * QD + B * N * N].reshape(B, N, N), out[B * QD + B * N * N:]
    f = engine.Usckf(B, nk=nk, nl=nl)
    f.set_state(sc["mu"], sc["P"])
    f.predict(engine.PM_USCKF_TEST, sc["u"], sc["dt"], sc["Qi"])
    f.update(engine.MM_USCKF_VO, sc["z"], sc["Ri"])
    np.testing.assert_array_equal(mu, f.mu())
    np.testing.assert_array_equal(P, f.P())
    np.testing.assert_array_equal(st, f.status())
    assert not st.any()
    # and the per-instance noise made a difference
    g = engine.Usckf(B, nk=nk, nl=nl)
    g.set_state(sc["mu"], sc["P"])
    g.predict(engine.PM_USCKF_TEST, sc["u"], sc["dt"], sc["Qi"][0])
    g.update(engine.MM_USCKF_VO, sc["z"], sc["Ri"][0])
    assert not np.array_equal(P, g.P())
