"""Storage of a batch: the UKF SoA arrays and the USCKF / MSCKF instance records (DESIGN §3).  Upload, download,
replication and the ensemble statistics address mu and P through one layout descriptor; these tests check every kind
and shape against plain numpy, bit for bit where nothing is computed."""
import numpy as np
import pytest

import parity
from slam_localization_b200 import engine, synth

pytestmark = pytest.mark.gpu
B = 203                  # ragged: a UKF batch pads its SoA rows to 224 instances
USCKF_SHAPES = [(3, 0), (3, 3), (3, 6), (3, 9), (6, 0), (6, 3), (6, 6), (9, 0), (9, 3)]

# name -> (batch factory, manifold blocks, feature scalars)
BATCHES = {"ukf_pose6": (lambda b: engine.Ukf(b, layout=engine.LAYOUT_POSE6), synth.LAYOUT_BLOCKS[6], 0),
           "ukf_mtk9": (lambda b: engine.Ukf(b, layout=engine.LAYOUT_MTK9), synth.LAYOUT_BLOCKS[9], 0)}
for _nk, _nl in USCKF_SHAPES:
    BATCHES["usckf_%d_%d" % (_nk, _nl)] = (lambda b, nk=_nk, nl=_nl: engine.Usckf(b, nk=nk, nl=nl),
                                           synth.STATE_BLOCKS * 3, _nk + _nl)
for _k in (1, 10):
    BATCHES["msckf_%d" % _k] = (lambda b, k=_k: engine.Msckf(b, nclones=k), synth.STATE_BLOCKS + [0, 1] * _k, 0)


def _inputs(name, n, seed):
    """n seeded means and n general (not symmetric) matrices: upload reads the lower triangle only."""
    _, blocks, nfeat = BATCHES[name]
    rng = np.random.default_rng(seed)
    mu = synth.random_q(rng, n, blocks, nfeat)
    N = 3 * len(blocks) + nfeat
    return mu, rng.normal(size=(n, N, N))


@pytest.mark.parametrize("name", list(BATCHES))
def test_upload_download_round_trip_is_bitwise(name):
    f = BATCHES[name][0](B)
    mu, P = _inputs(name, B, 401)
    f.set_state(mu, P)
    np.testing.assert_array_equal(f.mu(), mu)
    np.testing.assert_array_equal(f.P(), parity.symmetrize_lower(P))


@pytest.mark.parametrize("name", list(BATCHES))
def test_partial_transfers_touch_only_the_first_instances(name):
    k = 37
    f = BATCHES[name][0](B)
    mu, P = _inputs(name, B, 402)
    mu2, P2 = _inputs(name, k, 403)
    f.set_state(mu, P)
    check, lib = engine.check, engine.lib()
    check(lib.slb_upload(f.h, engine.FIELD_MU, engine._hp(mu2), mu2.size, engine._stream()))
    check(lib.slb_upload(f.h, engine.FIELD_P, engine._hp(P2), P2.size, engine._stream()))
    mu[:k], P[:k] = mu2, P2
    np.testing.assert_array_equal(f.mu(), mu)
    np.testing.assert_array_equal(f.P(), parity.symmetrize_lower(P))
    np.testing.assert_array_equal(f.mu(first=k), mu2)
    np.testing.assert_array_equal(f.P(first=k), parity.symmetrize_lower(P2))


@pytest.mark.parametrize("name", list(BATCHES))
def test_replicate_gives_instance_i_the_state_of_i_mod_k(name):
    k = 5
    f = BATCHES[name][0](B)
    mu, P = _inputs(name, k, 404)
    f.set_state(mu, P, replicate=True)
    idx = np.arange(B) % k
    np.testing.assert_array_equal(f.mu(), mu[idx])
    np.testing.assert_array_equal(f.P(), parity.symmetrize_lower(P)[idx])


def test_transfers_across_staging_chunks():
    """8192 (3,9) instances are 151 MB of dense covariances: upload and download run in three staging chunks."""
    n = 8192
    f = BATCHES["usckf_3_9"][0](n)
    mu, P = _inputs("usckf_3_9", n, 405)
    f.set_state(mu, P)
    np.testing.assert_array_equal(f.mu(), mu)
    np.testing.assert_array_equal(f.P(), parity.symmetrize_lower(P))
    k = 3
    f.set_state(mu[:k], P[:k], replicate=True)
    np.testing.assert_array_equal(f.P(), parity.symmetrize_lower(P[:k])[np.arange(n) % k])


def _vectorize(blocks, nfeat, mu):
    """(B, N) vectorised means: SO3 blocks by their logarithm, 2 atan(|qv| / qw) / |qv| qv, the rest as stored."""
    cols, o = [], 0
    for so3 in blocks:
        if so3:
            w, v = mu[:, o:o + 1], mu[:, o + 1:o + 4]
            nv = np.linalg.norm(v, axis=1, keepdims=True)
            cols.append(2.0 * np.arctan(nv / w) / nv * v)
            o += 4
        else:
            cols.append(mu[:, o:o + 3])
            o += 3
    cols.append(mu[:, o:o + nfeat])
    return np.concatenate(cols, axis=1)


@pytest.mark.parametrize("name", ["usckf_3_9", "msckf_10"])
def test_ensemble_stats_of_records_match_numpy(name):
    n = 3000
    factory, blocks, nfeat = BATCHES[name]
    f = factory(n)
    mu, P = _inputs(name, n, 406)
    f.set_state(mu, P)
    out = f.ensemble_stats().numpy()
    X = _vectorize(blocks, nfeat, mu)
    N = X.shape[1]
    assert out[0] == n
    np.testing.assert_allclose(out[1:1 + N], X.sum(0), rtol=1e-10, atol=1e-9)
    np.testing.assert_allclose(out[1 + N:].reshape(N, N), X.T @ X, rtol=1e-10, atol=1e-9)
