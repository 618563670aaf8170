// slb_core_next.cu -- SURVEY 8(f) rows f3 and f4, one instance per THREAD.  Compiled with -fmad=false.
//
//   f3  DataModel<double,3>::safeFusion(data2)                 src/core/DataModel.hpp:62-130
//   f4  DeadReckon::updateAttitude / updatePose (uncertain)    src/core/DeadReckon.hpp:246-286, 30-79
//       TransformWithUncertainty::operator*                    src/core/Transform.cpp:215-254 (+ helpers :35-138)
//
// These are the producers/consumers either side of the filters (odometry delta-pose with its 6x6 covariance
// feeding the MSCKF process model; fusion of 3-D estimates): tiny dense algebra (3x3 .. 6x6) per instance with
// 100-700 bytes of traffic, so the mapping is a thread per instance with everything in registers / local arrays,
// consecutive threads on consecutive instances.  Like DataModel::fusion the arithmetic follows the reference as
// written, operation by operation without FMA contraction: the third-party pieces are Eigen's published
// algorithms (two-sided JacobiSVD, Quaternion <-> Matrix3, AngleAxis(Quaternion), fixed-size 3x3 inverse by
// cofactors, LLT).  safeFusion keeps the reference's T = U2^T sqrt(D1) U1 (DataModel.hpp:106) as written.
#include <cfloat>

#include "slb_internal.h"
#include "slb_math.cuh"

namespace slbd {

// ---- tiny fixed-size dense helpers (row-major, fully unrolled) ---------------------------------------------
template <int R, int C>
struct Mx {
    double a[R * C];
    SLB_DEV double &operator()(int i, int j) { return a[i * C + j]; }
    SLB_DEV double operator()(int i, int j) const { return a[i * C + j]; }
    SLB_DEV void zero() {
#pragma unroll
        for (int e = 0; e < R * C; ++e) a[e] = 0.0;
    }
};
// C(i,j) = sum_k A(i,k) B(k,j), k ascending from 0.0 (the oracle's / Eigen's lazy-product order)
template <int R, int K, int C>
SLB_DEV Mx<R, C> mul(const Mx<R, K> &A, const Mx<K, C> &B) {
    Mx<R, C> O;
#pragma unroll
    for (int i = 0; i < R; ++i)
#pragma unroll
        for (int j = 0; j < C; ++j) {
            double s = 0.0;
#pragma unroll
            for (int k = 0; k < K; ++k) s += A(i, k) * B(k, j);
            O(i, j) = s;
        }
    return O;
}
template <int R, int C>
SLB_DEV Mx<C, R> tr(const Mx<R, C> &A) {
    Mx<C, R> O;
#pragma unroll
    for (int i = 0; i < R; ++i)
#pragma unroll
        for (int j = 0; j < C; ++j) O(j, i) = A(i, j);
    return O;
}
template <int R, int C>
SLB_DEV Mx<R, C> addm(const Mx<R, C> &A, const Mx<R, C> &B) {
    Mx<R, C> O;
#pragma unroll
    for (int e = 0; e < R * C; ++e) O.a[e] = A.a[e] + B.a[e];
    return O;
}
template <int R, int C>
SLB_DEV Mx<R, C> subm(const Mx<R, C> &A, const Mx<R, C> &B) {
    Mx<R, C> O;
#pragma unroll
    for (int e = 0; e < R * C; ++e) O.a[e] = A.a[e] - B.a[e];
    return O;
}
template <int R, int C>
SLB_DEV Mx<R, C> scl(const Mx<R, C> &A, double s) {
    Mx<R, C> O;
#pragma unroll
    for (int e = 0; e < R * C; ++e) O.a[e] = A.a[e] * s;
    return O;
}
template <int N>
SLB_DEV Mx<N, N> eye() {
    Mx<N, N> O;
    O.zero();
#pragma unroll
    for (int i = 0; i < N; ++i) O(i, i) = 1.0;
    return O;
}
template <int R, int C>
SLB_DEV void mulv(const Mx<R, C> &A, const double *x, double *y) {
#pragma unroll
    for (int i = 0; i < R; ++i) {
        double s = 0.0;
#pragma unroll
        for (int j = 0; j < C; ++j) s += A(i, j) * x[j];
        y[i] = s;
    }
}
// Eigen's fixed-size 3x3 inverse: cofactors / determinant
SLB_DEV Mx<3, 3> inv33(const Mx<3, 3> &A) {
    Mx<3, 3> C;
    auto cof = [&](int i, int j) {
        const int i1 = (i + 1) % 3, i2 = (i + 2) % 3, j1 = (j + 1) % 3, j2 = (j + 2) % 3;
        return A(i1, j1) * A(i2, j2) - A(i1, j2) * A(i2, j1);
    };
    const double c00 = cof(0, 0), c10 = cof(1, 0), c20 = cof(2, 0);
    const double det = c00 * A(0, 0) + c10 * A(1, 0) + c20 * A(2, 0);
    const double invdet = 1.0 / det;
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j) C(j, i) = cof(i, j) * invdet;
    return C;
}

// ---- Eigen::JacobiSVD<MatrixXd>(A, ComputeThinU), 3 x 3 real -------------------------------------------------
struct JRot { double c, s; };
SLB_DEV JRot make_jacobi(double x, double y, double z) {
    const double deno = 2.0 * fabs(y);
    if (deno < DBL_MIN) return {1.0, 0.0};
    const double tau = (x - z) / deno;
    const double w = sqrt(tau * tau + 1.0);
    const double t = tau > 0.0 ? 1.0 / (tau + w) : 1.0 / (tau - w);
    const double sign_t = t > 0.0 ? 1.0 : -1.0;
    const double n = 1.0 / sqrt(t * t + 1.0);
    return {n, -sign_t * (y / fabs(y)) * fabs(t) * n};
}
// pick3 is still used by rot_to_quat's largest-diagonal branch (runtime index through selects)
SLB_DEV double pick3(const Mx<3, 3> &M, int i, int j) {
    double v = M.a[0];
#pragma unroll
    for (int e = 1; e < 9; ++e) v = (i * 3 + j == e) ? M.a[e] : v;
    return v;
}
// One (p, q) step of a Jacobi sweep with compile-time indices: everything stays in named registers.
template <int P, int Q>
SLB_DEV void jacobi_pair(Mx<3, 3> &W, Mx<3, 3> &U, double &max_diag, bool &finished) {
    const double precision = 2.0 * DBL_EPSILON, consider_zero = DBL_MIN;
    const double thr = fmax(consider_zero, precision * max_diag);
    if (fabs(W(P, Q)) > thr || fabs(W(Q, P)) > thr) {
        finished = false;
        // internal::real_2x2_jacobi_svd
        double m00 = W(P, P), m01 = W(P, Q), m10 = W(Q, P), m11 = W(Q, Q);
        JRot rot1;
        const double t = m00 + m11, d = m10 - m01;
        if (fabs(d) < DBL_MIN) {
            rot1 = {1.0, 0.0};
        } else {
            const double u = t / d;
            const double tmp = sqrt(1.0 + u * u);
            rot1 = {u / tmp, 1.0 / tmp};
        }
        {
            const double a0 = rot1.c * m00 + rot1.s * m10, a1 = rot1.c * m01 + rot1.s * m11;
            const double b1 = -rot1.s * m01 + rot1.c * m11;
            m00 = a0; m01 = a1; m11 = b1;
        }
        const JRot jr = make_jacobi(m00, m01, m11);
        const JRot jrt = {jr.c, -jr.s};
        const JRot jl = {rot1.c * jrt.c - rot1.s * jrt.s, rot1.c * jrt.s + rot1.s * jrt.c};
        // m_workMatrix.applyOnTheLeft(p, q, j_left)
#pragma unroll
        for (int i = 0; i < 3; ++i) {
            const double x = W(P, i), y = W(Q, i);
            W(P, i) = jl.c * x + jl.s * y;
            W(Q, i) = -jl.s * x + jl.c * y;
        }
        // m_matrixU.applyOnTheRight(p, q, j_left.transpose()): rotates the columns with j_left
#pragma unroll
        for (int i = 0; i < 3; ++i) {
            const double x = U(i, P), y = U(i, Q);
            U(i, P) = jl.c * x + jl.s * y;
            U(i, Q) = -jl.s * x + jl.c * y;
        }
        // m_workMatrix.applyOnTheRight(p, q, j_right): rotates the columns with j_right^T
#pragma unroll
        for (int i = 0; i < 3; ++i) {
            const double x = W(i, P), y = W(i, Q);
            W(i, P) = jr.c * x - jr.s * y;
            W(i, Q) = jr.s * x + jr.c * y;
        }
        max_diag = fmax(max_diag, fmax(fabs(W(P, P)), fabs(W(Q, Q))));
    }
}
__device__ __noinline__ void jacobi_svd3(const Mx<3, 3> &A, Mx<3, 3> &U, double *sv) {
    double scale = 0.0;
#pragma unroll
    for (int e = 0; e < 9; ++e) scale = fmax(scale, fabs(A.a[e]));
    if (scale == 0.0) scale = 1.0;
    Mx<3, 3> W;
#pragma unroll
    for (int e = 0; e < 9; ++e) W.a[e] = A.a[e] / scale;
    U = eye<3>();
    double max_diag = fmax(fmax(fabs(W(0, 0)), fabs(W(1, 1))), fabs(W(2, 2)));
    bool finished = false;
    int guard = 0;
    while (!finished && guard++ < 64) {   // sweep order p = 1.., q < p: (1,0) (2,0) (2,1)
        finished = true;
        jacobi_pair<1, 0>(W, U, max_diag, finished);
        jacobi_pair<2, 0>(W, U, max_diag, finished);
        jacobi_pair<2, 1>(W, U, max_diag, finished);
    }
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        const double a = fabs(W(i, i));
        sv[i] = a;
        if (a != 0.0) {
            const double f = W(i, i) / a;
#pragma unroll
            for (int r = 0; r < 3; ++r) U(r, i) *= f;
        }
    }
#pragma unroll
    for (int i = 0; i < 3; ++i) sv[i] *= scale;
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        int pos = i;
#pragma unroll
        for (int k = 0; k < 3; ++k)
            if (k > i) {
                double sp = sv[0];
#pragma unroll
                for (int e = 1; e < 3; ++e) sp = pos == e ? sv[e] : sp;
                if (sv[k] > sp) pos = k;
            }
        double smax = sv[0];
#pragma unroll
        for (int e = 1; e < 3; ++e) smax = pos == e ? sv[e] : smax;
        if (smax == 0.0) break;
#pragma unroll
        for (int k = 0; k < 3; ++k)
            if (k > i && pos == k) {
                const double t = sv[i];
                sv[i] = sv[k];
                sv[k] = t;
#pragma unroll
                for (int r = 0; r < 3; ++r) {
                    const double u = U(r, i);
                    U(r, i) = U(r, k);
                    U(r, k) = u;
                }
            }
    }
}

__global__ void __launch_bounds__(128) safe_fusion_kernel(int64_t n, const double *x1, const double *C1, const double *x2, const double *C2,
                                                          double *xo, double *Co) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    Mx<3, 3> Ca, Cb;
    double a[3], b[3];
#pragma unroll
    for (int e = 0; e < 9; ++e) { Ca.a[e] = C1[i * 9 + e]; Cb.a[e] = C2[i * 9 + e]; }
#pragma unroll
    for (int e = 0; e < 3; ++e) { a[e] = x1[i * 3 + e]; b[e] = x2[i * 3 + e]; }
    const Mx<3, 3> I1 = inv33(Ca);
    Mx<3, 3> I2 = inv33(Cb);
    Mx<3, 3> U1, U2;
    double s1[3], s2[3];
    jacobi_svd3(I1, U1, s1);
    Mx<3, 3> sqrtD1;
    sqrtD1.zero();
#pragma unroll
    for (int k = 0; k < 3; ++k) sqrtD1(k, k) = sqrt(s1[k]);
    const Mx<3, 3> isq = inv33(sqrtD1);
    I2 = mul(mul(mul(mul(isq, tr(U1)), I2), U1), isq);  // :93
    jacobi_svd3(I2, U2, s2);
    const Mx<3, 3> T = mul(mul(tr(U2), sqrtD1), U1);  // :106 as written
    double d1[3], d2[3], res[3];
    mulv(T, a, d1);
    mulv(T, b, d2);
    Mx<3, 3> D3;
    D3.zero();
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        if (s2[k] < 1.0) { res[k] = d1[k]; D3(k, k) = 1.0; }
        else { res[k] = d2[k]; D3(k, k) = s2[k]; }
    }
    const Mx<3, 3> Ti = inv33(T);
    double xr[3];
    mulv(Ti, res, xr);
    const Mx<3, 3> Cr = mul(mul(Ti, inv33(D3)), tr(Ti));
#pragma unroll
    for (int e = 0; e < 3; ++e) xo[i * 3 + e] = xr[e];
#pragma unroll
    for (int e = 0; e < 9; ++e) Co[i * 9 + e] = Cr.a[e];
}

// ---- f4 ------------------------------------------------------------------------------------------------
SLB_DEV Mx<3, 3> quat_to_rot(const double *q) {
    const double w = q[0], x = q[1], y = q[2], z = q[3];
    const double tx = 2 * x, ty = 2 * y, tz = 2 * z;
    const double twx = tx * w, twy = ty * w, twz = tz * w;
    const double txx = tx * x, txy = ty * x, txz = tz * x;
    const double tyy = ty * y, tyz = tz * y, tzz = tz * z;
    Mx<3, 3> R;
    R(0, 0) = 1 - (tyy + tzz); R(0, 1) = txy - twz; R(0, 2) = txz + twy;
    R(1, 0) = txy + twz; R(1, 1) = 1 - (txx + tzz); R(1, 2) = tyz - twx;
    R(2, 0) = txz - twy; R(2, 1) = tyz + twx; R(2, 2) = 1 - (txx + tyy);
    return R;
}
SLB_DEV void rot_to_quat(const Mx<3, 3> &m, double *q) {
    double t = m(0, 0) + m(1, 1) + m(2, 2);
    if (t > 0.0) {
        t = sqrt(t + 1.0);
        q[0] = 0.5 * t;
        t = 0.5 / t;
        q[1] = (m(2, 1) - m(1, 2)) * t;
        q[2] = (m(0, 2) - m(2, 0)) * t;
        q[3] = (m(1, 0) - m(0, 1)) * t;
    } else {
        int i = 0;
        if (m(1, 1) > m(0, 0)) i = 1;
        if (m(2, 2) > pick3(m, i, i)) i = 2;
        const int j = (i + 1) % 3, k = (j + 1) % 3;
        t = sqrt(pick3(m, i, i) - pick3(m, j, j) - pick3(m, k, k) + 1.0);
        const double qi = 0.5 * t;
        t = 0.5 / t;
        q[0] = (pick3(m, k, j) - pick3(m, j, k)) * t;
        const double qj = (pick3(m, j, i) + pick3(m, i, j)) * t, qk = (pick3(m, k, i) + pick3(m, i, k)) * t;
#pragma unroll
        for (int e = 0; e < 3; ++e) q[1 + e] = e == i ? qi : (e == j ? qj : qk);
    }
}
SLB_DEV void q_to_r(const double *q, double *r) {
    double n = sqrt(q[1] * q[1] + q[2] * q[2] + q[3] * q[3]);
    if (n != 0.0) {
        const double angle = 2.0 * atan2(n, fabs(q[0]));
        if (q[0] < 0.0) n = -n;
#pragma unroll
        for (int i = 0; i < 3; ++i) r[i] = q[1 + i] / n * angle;
    } else {
        r[0] = 0.0; r[1] = 0.0; r[2] = 0.0;
    }
}
SLB_DEV Mx<3, 3> skew(const double *r) {
    Mx<3, 3> S;
    S.zero();
    S(0, 1) = -r[2]; S(0, 2) = r[1]; S(1, 0) = r[2]; S(1, 2) = -r[0]; S(2, 0) = -r[1]; S(2, 1) = r[0];
    return S;
}
SLB_DEV Mx<3, 3> outer3(const double *a, const double *b) {
    Mx<3, 3> M;
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j) M(i, j) = a[i] * b[j];
    return M;
}
SLB_DEV Mx<4, 3> dq_by_dr(const double *q) {
    double r[3];
    q_to_r(q, r);
    const double theta = sqrt(r[0] * r[0] + r[1] * r[1] + r[2] * r[2]);
    const double kappa = 0.5 - theta * theta / 48.0;
    const double lambda = 1.0 / 24.0 * (1.0 - theta * theta / 40.0);
    Mx<4, 3> res;
    const Mx<3, 3> rr = outer3(r, r);
#pragma unroll
    for (int j = 0; j < 3; ++j) res(0, j) = -q[1 + j] / 2.0;
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j) res(1 + i, j) = kappa * (i == j ? 1.0 : 0.0) - lambda * rr(i, j);
    return res;
}
SLB_DEV Mx<3, 4> dr_by_dq(const double *q) {
    const double mu = sqrt(q[1] * q[1] + q[2] * q[2] + q[3] * q[3]);
    const double sg = q[0] > 0 ? 1.0 : -1.0;
    const double tau = 2.0 * sg * (1.0 + mu * mu / 6.0);
    const double nu = -2.0 * sg * (2.0 / 3.0 + mu * mu / 5.0);
    Mx<3, 4> res;
    const Mx<3, 3> vv = outer3(q + 1, q + 1);
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        res(i, 0) = -2 * q[1 + i];
#pragma unroll
        for (int j = 0; j < 3; ++j) res(i, 1 + j) = tau * (i == j ? 1.0 : 0.0) + nu * vv(i, j);
    }
    return res;
}
SLB_DEV Mx<4, 4> dq2q1_by(const double *q, double sgn) {
    Mx<4, 4> res;
    res.zero();
    const Mx<3, 3> S = skew(q + 1);
#pragma unroll
    for (int j = 0; j < 3; ++j) { res(0, 1 + j) = -q[1 + j]; res(1 + j, 0) = q[1 + j]; }
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j) res(1 + i, 1 + j) = sgn * S(i, j);
    Mx<4, 4> out;
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) out(i, j) = (i == j ? 1.0 : 0.0) * q[0] + res(i, j);
    return out;
}
SLB_DEV Mx<3, 3> drx_by_dr(const double *q, const double *x) {
    double r[3];
    q_to_r(q, r);
    const double theta = sqrt(r[0] * r[0] + r[1] * r[1] + r[2] * r[2]);
    const double alpha = 1.0 - theta * theta / 6.0;
    const double beta = 0.5 - theta * theta / 24.0;
    const double gamma = 1.0 / 3.0 - theta * theta / 30.0;
    const double delta = -1.0 / 12.0 + theta * theta / 180.0;
    const Mx<3, 3> rr = outer3(r, r), Sx = skew(x), Sr = skew(r), I = eye<3>();
    const Mx<3, 3> A = addm(subm(scl(rr, gamma), scl(Sr, beta)), scl(I, alpha));
    const Mx<3, 3> B = addm(scl(rr, delta), scl(I, 2.0 * beta));
    return subm(mul(scl(Sx, -1.0), A), mul(mul(Sr, Sx), B));
}

// result = t2 * t1 (Transform.cpp:215-254); poses are pos(3) quat(w,x,y,z), covariances 6x6 over [r t]
// cov2 / cov1 / cov_out point at row-major 6x6 matrices in global memory: 3x3 blocks are fetched and stored on demand, so
// no 6x6 matrix is ever live in registers.
SLB_DEV void transform_compose(const double *pose2, const double *cov2, const double *pose1, const double *cov1, double *pose_out,
                               double *cov_out) {
    const Mx<3, 3> R1 = quat_to_rot(pose1 + 3), R2 = quat_to_rot(pose2 + 3);
    double q1[4], q2[4], q[4];
    rot_to_quat(R1, q1);
    rot_to_quat(R2, q2);
    quat_mul(q2, q1, q);
    // J1 = [A1 0; 0 R2], J2 = [A2 0; B2 I] (Transform.cpp:233-247): the two 6x6 sandwiches J c J^T are evaluated on
    // their 3x3 blocks.  The skipped terms are exact zeros of the dense products, so the sums (and their order) are the
    // reference's; half the multiplications and a third of the live registers of the dense form.
    {
        const Mx<3, 4> a = dr_by_dq(q);
        const Mx<3, 3> A1 = mul(mul(a, dq2q1_by(q2, 1.0)), dq_by_dr(q1));
        const Mx<3, 3> A2 = mul(mul(a, dq2q1_by(q1, -1.0)), dq_by_dr(q2));
        const Mx<3, 3> B2 = drx_by_dr(q2, pose1);
        auto blk = [](const double *c, int bi, int bj) {
            Mx<3, 3> o;
#pragma unroll
            for (int i = 0; i < 3; ++i)
#pragma unroll
                for (int j = 0; j < 3; ++j) o(i, j) = c[(3 * bi + i) * 6 + 3 * bj + j];
            return o;
        };
        auto put = [&](int bi, int bj, const Mx<3, 3> &x, const Mx<3, 3> &y) {
#pragma unroll
            for (int i = 0; i < 3; ++i)
#pragma unroll
                for (int j = 0; j < 3; ++j) cov_out[(3 * bi + i) * 6 + 3 * bj + j] = x(i, j) + y(i, j);
        };
        const Mx<3, 3> A1t = tr(A1), A2t = tr(A2), B2t = tr(B2), R2t = tr(R2);
        // (J1 c1) blocks and (J2 c2) blocks
        const Mx<3, 3> p_rr = mul(A1, blk(cov1, 0, 0)), p_rt = mul(A1, blk(cov1, 0, 1));
        const Mx<3, 3> p_tr = mul(R2, blk(cov1, 1, 0)), p_tt = mul(R2, blk(cov1, 1, 1));
        const Mx<3, 3> c2rr = blk(cov2, 0, 0), c2rt = blk(cov2, 0, 1);
        const Mx<3, 3> s_rr = mul(A2, c2rr), s_rt = mul(A2, c2rt);
        const Mx<3, 3> s_tr = addm(mul(B2, c2rr), blk(cov2, 1, 0)), s_tt = addm(mul(B2, c2rt), blk(cov2, 1, 1));
        put(0, 0, mul(p_rr, A1t), mul(s_rr, A2t));
        put(0, 1, mul(p_rt, R2t), addm(mul(s_rr, B2t), s_rt));
        put(1, 0, mul(p_tr, A1t), mul(s_tr, A2t));
        put(1, 1, mul(p_tt, R2t), addm(mul(s_tr, B2t), s_tt));
    }
    const Mx<3, 3> R = mul(R2, R1);
#pragma unroll
    for (int i = 0; i < 3; ++i) pose_out[i] = R2(i, 0) * pose1[0] + R2(i, 1) * pose1[1] + R2(i, 2) * pose1[2] + pose2[i];
    rot_to_quat(R, pose_out + 3);
}

__global__ void __launch_bounds__(64) transform_compose_kernel(int64_t n, const double *pose2, const double *cov2, const double *pose1,
                                                               const double *cov1, double *pose_out, double *cov_out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    double p2[7], p1[7], po[7];
#pragma unroll
    for (int e = 0; e < 7; ++e) { p2[e] = pose2[i * 7 + e]; p1[e] = pose1[i * 7 + e]; }
    transform_compose(p2, cov2 + i * 36, p1, cov1 + i * 36, po, cov_out + i * 36);
#pragma unroll
    for (int e = 0; e < 7; ++e) pose_out[i * 7 + e] = po[e];
}

// DeadReckon::updateAttitude (DeadReckon.hpp:246-286)
SLB_DEV void dr_update_attitude(double dt, const double *w0, const double *w1, double *dq) {
    auto omega = [](const double *w) {
        Mx<4, 4> O;
        O.zero();
        O(0, 1) = -w[0]; O(0, 2) = -w[1]; O(0, 3) = -w[2];
        O(1, 0) = w[0]; O(1, 2) = w[2]; O(1, 3) = -w[1];
        O(2, 0) = w[1]; O(2, 1) = -w[2]; O(2, 3) = w[0];
        O(3, 0) = w[2]; O(3, 1) = w[1]; O(3, 2) = -w[0];
        return O;
    };
    const Mx<4, 4> O4 = omega(w0), Oo = omega(w1), I = eye<4>();
    const double n2 = w0[0] * w0[0] + w0[1] * w0[1] + w0[2] * w0[2];
    const double dt2 = dt * dt, dt3 = dt * dt * dt;  // the reference writes pow(dt,2), pow(dt,3): equal to these products up to an ulp
    Mx<4, 4> M = addm(I, scl(scl(O4, 0.75), dt));
    M = subm(M, scl(scl(Oo, 0.25), dt));
    M = subm(M, scl(I, (1.0 / 6.0) * n2 * dt2));
    M = subm(M, scl(mul(scl(O4, 1.0 / 24.0), Oo), dt2));
    M = subm(M, scl(scl(O4, (1.0 / 48.0) * n2), dt3));
    const double quat[4] = {M(0, 0), M(1, 0), M(2, 0), M(3, 0)};
    const double n = sqrt(quat[0] * quat[0] + quat[1] * quat[1] + quat[2] * quat[2] + quat[3] * quat[3]);
#pragma unroll
    for (int i = 0; i < 4; ++i) dq[i] = quat[i] / n;
}

// unblocked LLT of a 6x6 whose off-diagonal 3x3 blocks are zero, then L L^T (DeadReckon.hpp:50-52)
SLB_DEV Mx<6, 6> llt_llt6(const Mx<6, 6> &A) {
    Mx<6, 6> L;
    L.zero();
#pragma unroll
    for (int k = 0; k < 6; ++k) {
        double x = A(k, k);
#pragma unroll
        for (int p = 0; p < 6; ++p)
            if (p < k) x -= L(k, p) * L(k, p);
        x = sqrt(x);
        L(k, k) = x;
#pragma unroll
        for (int i = 0; i < 6; ++i)
            if (i > k) {
                double s = A(i, k);
#pragma unroll
                for (int p = 0; p < 6; ++p)
                    if (p < k) s -= L(i, p) * L(k, p);
                L(i, k) = s / x;
            }
    }
    return mul(L, tr(L));
}

__global__ void __launch_bounds__(64) dr_update_pose_kernel(int64_t n, double dt, const double *vel0, const double *vel1, const double *velcov,
                                                            const double *prev_pose, const double *prev_cov, double *post_pose,
                                                            double *post_cov, double *delta_pose, double *delta_cov) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    double v0[6], v1[6], pp[7], dp[7], po[7];
#pragma unroll
    for (int e = 0; e < 6; ++e) { v0[e] = vel0[i * 6 + e]; v1[e] = vel1[i * 6 + e]; }
#pragma unroll
    for (int e = 0; e < 7; ++e) pp[e] = prev_pose[i * 7 + e];
    dr_update_attitude(dt, v0 + 3, v1 + 3, dp + 3);
#pragma unroll
    for (int e = 0; e < 3; ++e) dp[e] = (dt / 2.0) * (v0[e] + v1[e]);
    Mx<6, 6> dc;
    dc.zero();
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            dc(r, c) = __ldg(velcov + (3 + r) * 6 + 3 + c) * dt * dt;
            dc(3 + r, 3 + c) = __ldg(velcov + r * 6 + c) * dt * dt;
        }
    {   // deltaPose's covariance goes to its output array first; the composition reads it back block by block
        const Mx<6, 6> dcov = llt_llt6(dc);
#pragma unroll
        for (int e = 0; e < 36; ++e) delta_cov[i * 36 + e] = dcov.a[e];
    }
    transform_compose(pp, prev_cov + i * 36, dp, delta_cov + i * 36, po, post_cov + i * 36);
#pragma unroll
    for (int e = 0; e < 7; ++e) { post_pose[i * 7 + e] = po[e]; delta_pose[i * 7 + e] = dp[e]; }
}

}  // namespace slbd

using namespace slb;

extern "C" {

int slb_datamodel_safe_fuse(int64_t n, const double *x1, const double *C1, const double *x2, const double *C2, double *xo, double *Co,
                            void *stream) {
    if (n < 0 || !x1 || !C1 || !x2 || !C2 || !xo || !Co) return set_error(SLB_ERR_INVALID, "slb_datamodel_safe_fuse: bad argument");
    if (n == 0) return SLB_OK;
    if (need_device("slb_datamodel_safe_fuse: no CUDA device (this engine has no CPU fallback)") != SLB_OK) return SLB_ERR_NO_DEVICE;
    return launch(slbd::safe_fusion_kernel, (unsigned)((n + 127) / 128), 128, 0, (cudaStream_t)stream, n, x1, C1, x2, C2, xo, Co);
}

int slb_transform_compose(int64_t n, const double *pose2, const double *cov2, const double *pose1, const double *cov1, double *pose_out,
                          double *cov_out, void *stream) {
    if (n < 0 || !pose2 || !cov2 || !pose1 || !cov1 || !pose_out || !cov_out)
        return set_error(SLB_ERR_INVALID, "slb_transform_compose: bad argument");
    if (n == 0) return SLB_OK;
    if (need_device("slb_transform_compose: no CUDA device (this engine has no CPU fallback)") != SLB_OK) return SLB_ERR_NO_DEVICE;
    return launch(slbd::transform_compose_kernel, (unsigned)((n + 63) / 64), 64, 0, (cudaStream_t)stream, n, pose2, cov2, pose1,
                  cov1, pose_out, cov_out);
}

int slb_deadreckon_update_pose(int64_t n, double dt, const double *vel0, const double *vel1, const double *velcov, const double *prev_pose,
                               const double *prev_cov, double *post_pose, double *post_cov, double *delta_pose, double *delta_cov,
                               void *stream) {
    if (n < 0 || !vel0 || !vel1 || !velcov || !prev_pose || !prev_cov || !post_pose || !post_cov || !delta_pose || !delta_cov)
        return set_error(SLB_ERR_INVALID, "slb_deadreckon_update_pose: bad argument");
    if (n == 0) return SLB_OK;
    if (need_device("slb_deadreckon_update_pose: no CUDA device (this engine has no CPU fallback)") != SLB_OK) return SLB_ERR_NO_DEVICE;
    return launch(slbd::dr_update_pose_kernel, (unsigned)((n + 63) / 64), 64, 0, (cudaStream_t)stream, n, dt, vel0, vel1, velcov,
                  prev_pose, prev_cov, post_pose, post_cov, delta_pose, delta_cov);
}

}  // extern "C"
