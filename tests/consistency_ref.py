"""Numpy restatement of the Mahalanobis distance m2 = nu^T S^-1 nu that the UKFoM and USCKF updates hand to their gate
(ukfom::ukf::update / Usckf::update, Usckf.hpp:260-294; oracle/slo_filters.hpp Ukf::update, Usckf::update), and of NEES,
for the NIS capture and consistency tests.  Vectorised over the sigma points of one instance: sigma point 2j+1 / 2j+2 is
mu [+] +-L(:, j) with L the lower Cholesky factor of P, sigma point 0 is mu."""
import numpy as np

from slam_localization_b200 import synth

CHI2_5 = [0.0, 3.84, 5.99, 7.81, 9.49, 11.07, 12.59, 14.07, 15.51, 16.92]   # Usckf.hpp:794-855


def _deltas(P):
    L = np.linalg.cholesky(P)
    n = P.shape[0]
    D = np.zeros((2 * n + 1, n))
    D[1::2] = L.T
    D[2::2] = -L.T
    return D


def _m2(Z, z, R):
    zb = Z.mean(axis=0)
    DZ = Z - zb
    S = 0.5 * DZ.T @ DZ + R
    nu = z - zb
    return float(nu @ np.linalg.solve(S, nu))


def ukf_m2(mu, P, z, R):
    """One UKFoM instance with the GPS position model (z = pos): m2 of its update."""
    D = _deltas(P)
    return _m2(mu[0:3] + D[:, 0:3], z, R)


def usckf_m2(nk, mu, P, z, R):
    """One USCKF instance with the VO model of test/UsckfUnitTest.cpp:62-86: m2 of its update."""
    D = _deltas(P)
    pk = mu[0:3] + D[:, 0:3]
    qk = synth._qmul(np.broadcast_to(mu[3:7], (len(D), 4)), synth._qexp(D[:, 3:6]))
    pi = mu[26:29] + D[:, 24:27]
    qi = synth._qmul(np.broadcast_to(mu[29:33], (len(D), 4)), synth._qexp(D[:, 27:30]))
    qc = qi * np.array([1.0, -1.0, -1.0, -1.0])
    dq = synth._qmul(qc, qk)
    f = mu[39:39 + nk] + D[:, 36:36 + nk]
    Z = np.concatenate([synth._qrot(dq, f[:, c:c + 3]) + (pk - pi) for c in range(0, nk, 3)], axis=1)
    return _m2(Z, z, R)


def so3_log(q):
    """Rotation vector of unit quaternions (..., 4) (w, x, y, z)."""
    q = np.where(q[..., :1] < 0, -q, q)
    nv = np.linalg.norm(q[..., 1:], axis=-1, keepdims=True)
    th = 2.0 * np.arctan2(nv, q[..., :1])
    return np.where(nv > 1e-15, th / np.maximum(nv, 1e-300), 2.0) * q[..., 1:]


def tangent_error(blocks, nfeat, truth, mu):
    """truth [-] mu, (B, 3 nblk + nfeat): log(mu_q^-1 truth_q) on SO3 blocks, a difference elsewhere."""
    out, o = [], 0
    for s in blocks:
        if s:
            qc = mu[:, o:o + 4] * np.array([1.0, -1.0, -1.0, -1.0])
            out.append(so3_log(synth._qmul(qc, truth[:, o:o + 4])))
            o += 4
        else:
            out.append(truth[:, o:o + 3] - mu[:, o:o + 3])
            o += 3
    out.append(truth[:, o:o + nfeat] - mu[:, o:o + nfeat])
    return np.concatenate(out, axis=1)


def boxplus(blocks, nfeat, mu, d):
    """mu [+] d for (B, qdim) / (B, 3 nblk + nfeat)."""
    out, o = [], 0
    for b, s in enumerate(blocks):
        if s:
            out.append(synth._qmul(mu[:, o:o + 4], synth._qexp(d[:, 3 * b:3 * b + 3])))
            o += 4
        else:
            out.append(mu[:, o:o + 3] + d[:, 3 * b:3 * b + 3])
            o += 3
    out.append(mu[:, o:o + nfeat] + d[:, 3 * len(blocks):])
    return np.concatenate(out, axis=1)


def nees(blocks, nfeat, truth, mu, P, t0, n):
    """e_sub^T P_sub^-1 e_sub per instance (numpy solve)."""
    e = tangent_error(blocks, nfeat, truth, mu)[:, t0:t0 + n]
    Ps = P[:, t0:t0 + n, t0:t0 + n]
    return np.einsum("bi,bi->b", e, np.linalg.solve(Ps, e[..., None])[..., 0])
