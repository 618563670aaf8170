"""NIS capture and consistency statistics through the host C++ facade: tests/facade_consistency_test.cpp runs one USCKF
predict + update with capture on, then mahalanobis() and consistencyStats(); its results must be the Python engine's,
bit for bit.  Without a GPU the binary must refuse to compute."""
import os
import subprocess

import numpy as np
import pytest

from slam_localization_b200 import build as slb_build
from slam_localization_b200 import engine, synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EXE = os.path.join(ROOT, "tests", "_build", "facade_consistency_test")


def _build():
    slb_build.build()
    os.makedirs(os.path.dirname(EXE), exist_ok=True)
    src = os.path.join(ROOT, "tests", "facade_consistency_test.cpp")
    hdr = os.path.join(ROOT, "slam-localization_b200", "facade", "localization_b200.hpp")
    if not os.path.exists(EXE) or os.path.getmtime(EXE) < max(os.path.getmtime(src), os.path.getmtime(hdr)):
        csrc = os.path.join(ROOT, "slam-localization_b200", "csrc")
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-o", EXE, src, "-L" + csrc, "-lslb", "-Wl,-rpath," + csrc,
                               "-L/usr/local/cuda/lib64", "-Wl,-rpath,/usr/local/cuda/lib64"])
    return EXE


def _scenario(B, seed=801):
    sc = synth.usckf_scenario(B, seed=seed)
    rng = np.random.default_rng(seed + 1)
    sc["truth"] = sc["mu"].copy()
    sc["truth"][:, 0:3] += 0.01 * rng.normal(size=(B, 3))
    sc["truth"][:, 26:29] += 0.01 * rng.normal(size=(B, 3))
    return sc


def _run(tmp_path, sc, B, nk=3, nl=9):
    fin, fout = str(tmp_path / "in.bin"), str(tmp_path / "out.bin")
    parts = [np.array([B, nk, nl, sc["dt"]], float), sc["mu"], sc["P"], sc["u"], sc["Q"], sc["z"], sc["R"], sc["truth"]]
    np.concatenate([np.ravel(p) for p in parts]).astype(np.float64).tofile(fin)
    p = subprocess.run([_build(), fin, fout], capture_output=True, text=True)
    return p, fout


def test_facade_consistency_driver_compiles_and_refuses_without_gpu(tmp_path):
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present: covered by the GPU test below")
    p, _ = _run(tmp_path, _scenario(4), 4)
    assert p.returncode == 3 and "NO_DEVICE" in p.stdout


@pytest.mark.gpu
def test_facade_consistency_equals_engine(tmp_path):
    B = 37
    sc = _scenario(B)
    p, fout = _run(tmp_path, sc, B)
    assert p.returncode == 0 and "MSCKF_REFUSED" in p.stdout and "OK" in p.stdout, p.stdout + p.stderr
    out = np.fromfile(fout, dtype=np.float64)
    nis, full, si = out[:B], out[B:B + 6], out[B + 6:B + 12]
    f = engine.Usckf(B)
    f.set_state(sc["mu"], sc["P"])
    f.set_nis_capture(True)
    f.predict(engine.PM_USCKF_TEST, sc["u"], sc["dt"], sc["Q"])
    f.update(engine.MM_USCKF_VO, sc["z"], sc["R"])
    np.testing.assert_array_equal(nis, f.nis())
    assert np.isfinite(nis).all()
    np.testing.assert_allclose(full, f.consistency_stats(sc["truth"]), rtol=1e-12)
    np.testing.assert_allclose(si, f.consistency_stats(sc["truth"], 24, 12), rtol=1e-12)
    assert full[0] == B and full[3] == B
