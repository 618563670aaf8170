// slb_math.cuh -- device-side manifold algebra and small dense FP64 helpers (sm_100a).
//
// Same maths as the reference's MTK SO3/vect blocks (State.hpp:186-200 via MTK::SO3::boxplus /
// boxminus / exp / log) and the Eigen routines its filters call; written for registers:
// every loop is fully unrolled over compile-time layouts so arrays never leave the register file.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace slbd {

#define SLB_DEV __device__ __forceinline__
#define SLB_HD __host__ __device__ __forceinline__

// ---- compile-time manifold layout: NB blocks of 3 DOF, bit b of MASK set = block b is SO3 ------
template <int NB_, unsigned MASK_>
struct Layout {
    static constexpr int NB = NB_;
    static constexpr unsigned MASK = MASK_;
    static constexpr int N = 3 * NB_;
    static constexpr int NP = N * (N + 1) / 2;  // packed lower triangle
    SLB_HD static constexpr bool so3(int b) { return (MASK_ >> b) & 1u; }
    SLB_HD static constexpr int qoff(int b) {
        int o = 0;
        for (int i = 0; i < b; ++i) o += ((MASK_ >> i) & 1u) ? 4 : 3;
        return o;
    }
    static constexpr int QD = qoff(NB_);
};
typedef Layout<2, 0x2> LayPose6;    // vect3 pos, SO3 orient            (SensorState)
typedef Layout<3, 0x2> LayMtk9;     // pos, orient, vel                 (mtk_state)
typedef Layout<4, 0x2> LayState12;  // pos, orient, velo, angvelo       (State)

SLB_HD constexpr int tri(int i, int j) { return i * (i + 1) / 2 + j; }  // i >= j
// row r of the packed index e = tri(r, c) (the column is then e - tri(r, 0)): a float square-root estimate and a +-1
// fix-up, exact for e < 2^20
SLB_DEV int tri_row(int e) {
    int r = (int)((sqrtf(8.0f * e + 1.0f) - 1.0f) * 0.5f);
    r += (tri(r + 1, 0) <= e) - (tri(r, 0) > e);
    return r;
}

// Offset of P(i, j), i >= j, in a USCKF record of dimension N: the lower block triangle of 8 x 8 tiles, tile rows in
// order, within a tile row the off-diagonal tiles first (row-major, 8 columns each), then the diagonal tile (its packed
// lower triangle).  The last tile row holds only its h = N - 8 (ceil(N / 8) - 1) live rows (h x 8 tiles, an h-row
// triangle), so tile row I starts where packed row 8 I would, at tri(8 I, 0), and the record is N (N + 1) / 2 doubles
// like the packed triangle.  Row-major inside a tile is the DMMA m8n8k4 accumulator order: lane 4 b + a holds entries
// (b, 2 a), (b, 2 a + 1) of a tile, i.e. doubles 2 lane and 2 lane + 1 of an off-diagonal tile, one aligned 16-byte
// access.  (MSCKF records and UKF arrays keep the packed row-major triangle, tri().)
SLB_HD constexpr int prec(int N, int i, int j) {
    const int I = i >> 3, J = j >> 3, h = N - 8 * I < 8 ? N - 8 * I : 8;
    return tri(8 * I, 0) + 8 * h * J + (J < I ? 8 * (i & 7) + (j & 7) : tri(i & 7, j & 7));
}

// How a batch is stored (DESIGN §3), filled once by slb_create.  The filter kernels fix their format at compile time;
// the host-launched utilities (transfers, replication, ensemble statistics, the sigma-point check) address the mean and
// the covariance only through mu() and P().
struct BatchLayout {
    int N, QD, NP;                // tangent dimension, q-vector length, N (N + 1) / 2
    int stride;                   // SoA row length: instances rounded up to 32
    int qstride, pstride;         // doubles per mean / covariance record (QD rounded up to 2, NP to 16)
    bool soa;                     // UKF: mu[c][stride], P[tri(r, c)][stride].  Otherwise instance records
    bool tiled;                   // USCKF records: P(r, c) at prec(N, r, c).  MSCKF records: at tri(r, c)
    int nblk;                     // manifold: 3-DOF blocks ...
    unsigned long long so3mask;   // ... block b is SO3 (4 doubles in the q-vector) if bit b is set, else vect3 ...
    int nfeat;                    // ... then this many plain feature scalars
    // offset of mean scalar c of instance i
    SLB_HD constexpr size_t mu(int i, int c) const { return soa ? (size_t)c * stride + i : (size_t)i * qstride + c; }
    // offset of P(r, c), r >= c, of instance i
    SLB_HD constexpr size_t P(int i, int r, int c) const {
        const int e = tiled ? prec(N, r, c) : tri(r, c);
        return soa ? (size_t)e * stride + i : (size_t)i * pstride + e;
    }
    // doubles of the mean / covariance storage of a batch of B instances
    SLB_HD constexpr size_t mu_size(int B) const { return soa ? (size_t)QD * stride : (size_t)B * qstride; }
    SLB_HD constexpr size_t P_size(int B) const { return soa ? (size_t)NP * stride : (size_t)B * pstride; }
};

// ---- SO3 -----------------------------------------------------------------------------------------
// Sigma-point deviations are small rotations, so exp / log almost always see small arguments.  Both
// have a branch-free polynomial fast path (minimax fits, relative error < 5e-18 before rounding) that
// replaces sqrt + sincos + div (exp) and sqrt + atan + 2 div (log) by ~15 DFMA; large arguments fall
// back to the libm formulation of MTK.  Either path is within a few ulp of the CPU oracle's glibc
// result -- far inside the 1e-9 parity tolerance.
// 1/w for finite, normal, non-zero w: MUFU.RCP64H seed + two Newton steps (full double accuracy,
// not correctly rounded; never used where the oracle comparison is bit-exact).
SLB_DEV double rcp_fast(double w) {
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(w));
    double e = fma(-w, r, 1.0);
    r = fma(r, e, r);
    e = fma(-w, r, 1.0);
    r = fma(r, e, r);
    return r;
}
// sqrt(x) and 1/sqrt(x) for x > 0 from the MUFU.RSQ64H seed and two Newton steps (full double
// accuracy, ~1 ulp; not the IEEE-rounded sqrt/div pair of the CPU oracle -- parity is at 1e-9).
SLB_DEV void sqrt_rsqrt(double x, double &s, double &rs) {
    double y;
    asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(x));
    double e = fma(-(x * y), y, 1.0);
    y = fma(0.5 * y, e, y);
    e = fma(-(x * y), y, 1.0);
    y = fma(0.5 * y, e, y);
    double r = x * y;
    r = fma(fma(-r, r, x), 0.5 * y, r);
    s = r;
    rs = y;
}

// 1/sqrt(x) alone (same seed and Newton steps as sqrt_rsqrt)
SLB_DEV double rsqrt_fast(double x) {
    double y;
    asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(x));
    double e = fma(-(x * y), y, 1.0);
    y = fma(0.5 * y, e, y);
    e = fma(-(x * y), y, 1.0);
    y = fma(0.5 * y, e, y);
    return y;
}

// MTK cos_sinc_sqrt: c = cos(sqrt(x)), s = sin(sqrt(x))/sqrt(x)
SLB_DEV void cos_sinc_sqrt(double x, double &c, double &s) {
    if (x < 1.0) {  // |rotation| < 2 rad
        // minimax fits on [0, 1], Estrin form (short dependency chains: the kernels are latency-, not issue-bound)
        const double cx2 = x * x;
        const double ct1_0 = fma(fma(-1.38888888888883668e-03, x, 4.16666666666666644e-02), cx2, fma(-5.00000000000000000e-01, x, 1.00000000000000000e+00));
        const double ct1_1 = fma(fma(-1.14694398696376668e-11, x, 2.08767438008076401e-09), cx2, fma(-2.75573191463304794e-07, x, 2.48015873013186193e-05));
        const double cx4 = cx2 * cx2;
        const double ct2_0 = fma(ct1_1, cx4, ct1_0);
        const double cx8 = cx4 * cx4;
        const double ct3_0 = fma(4.70967686713015879e-14, cx8, ct2_0);
        const double st1_0 = fma(fma(-1.98412698410874757e-04, x, 8.33333333333310597e-03), cx2, fma(-1.66666666666666657e-01, x, 1.00000000000000000e+00));
        const double st1_1 = fma(fma(-7.53548806448761316e-13, x, 1.60572333370398622e-10), cx2, fma(-2.50520930836997243e-08, x, 2.75573191523091937e-06));
        const double st2_0 = fma(st1_1, cx4, st1_0);
        c = ct3_0;
        s = st2_0;
    } else {
        const double sx = sqrt(x);
        double sn, cs;
        sincos(sx, &sn, &cs);
        c = cs;
        s = sn / sx;
    }
}
// exp(v, scale): (w,x,y,z) of a rotation by scale*|v| about v/|v|
SLB_DEV void so3_exp(const double v[3], double scale, double q[4]) {
    const double h = 0.5 * scale;
    const double n2 = v[0] * v[0] + v[1] * v[1] + v[2] * v[2];
    double c, s;
    cos_sinc_sqrt(h * h * n2, c, s);
    const double m = s * h;
    q[0] = c; q[1] = m * v[0]; q[2] = m * v[1]; q[3] = m * v[2];
}
// log(q) = 2 atan(|qv|/qw)/|qv| qv   (atan: +-q identified; |qv| clamped at 1e-11)
SLB_DEV void so3_log(const double q[4], double v[3]) {
    const double nv2 = q[1] * q[1] + q[2] * q[2] + q[3] * q[3];
    const double w = q[0];
    double s;
    if (nv2 <= 0.16 * (w * w)) {  // |qv|/|qw| <= 0.4: rotation below ~43 degrees
        // 2 atan(t)/(t |qw|) sign(qw) = (2/qw) f(t^2),  f(x) = atan(sqrt x)/sqrt x
        const double r = rcp_fast(w);
        const double x = nv2 * (r * r);  // minimax fit of f on [0, 0.16], Estrin form
        const double ax2 = x * x;
        const double at1_0 = fma(fma(-1.42857142821344346e-01, x, 1.99999999999695866e-01), ax2, fma(-3.33333333333332316e-01, x, 1.00000000000000000e+00));
        const double at1_1 = fma(fma(-6.66392574614696059e-02, x, 7.69212730997153177e-02), ax2, fma(-9.09090122859413791e-02, x, 1.11111108929975527e-01));
        const double at1_2 = fma(fma(-1.88731700307688370e-02, x, 3.88960642020704864e-02), ax2, fma(-5.07008289291807218e-02, x, 5.85429330706751586e-02));
        const double ax4 = ax2 * ax2;
        const double at2_0 = fma(at1_1, ax4, at1_0);
        const double ax8 = ax4 * ax4;
        const double at3_0 = fma(at1_2, ax8, at2_0);
        s = (r + r) * at3_0;
    } else {
        double nv = sqrt(nv2);
        nv = nv < 1e-11 ? 1e-11 : nv;
        s = 2.0 / nv * atan(nv / w);
    }
    v[0] = s * q[1]; v[1] = s * q[2]; v[2] = s * q[3];
}
SLB_DEV void quat_mul(const double a[4], const double b[4], double o[4]) {
    const double w = a[0] * b[0] - a[1] * b[1] - a[2] * b[2] - a[3] * b[3];
    const double x = a[0] * b[1] + a[1] * b[0] + a[2] * b[3] - a[3] * b[2];
    const double y = a[0] * b[2] + a[2] * b[0] + a[3] * b[1] - a[1] * b[3];
    const double z = a[0] * b[3] + a[3] * b[0] + a[1] * b[2] - a[2] * b[1];
    o[0] = w; o[1] = x; o[2] = y; o[3] = z;
}
// conj(a) * b
SLB_DEV void quat_cmul(const double a[4], const double b[4], double o[4]) {
    const double w = a[0] * b[0] + a[1] * b[1] + a[2] * b[2] + a[3] * b[3];
    const double x = a[0] * b[1] - a[1] * b[0] - a[2] * b[3] + a[3] * b[2];
    const double y = a[0] * b[2] - a[2] * b[0] - a[3] * b[1] + a[1] * b[3];
    const double z = a[0] * b[3] - a[3] * b[0] - a[1] * b[2] + a[2] * b[1];
    o[0] = w; o[1] = x; o[2] = y; o[3] = z;
}
// q * v (Eigen _transformVector form)
SLB_DEV void quat_rotate(const double q[4], const double v[3], double o[3]) {
    const double tx = 2.0 * (q[2] * v[2] - q[3] * v[1]);
    const double ty = 2.0 * (q[3] * v[0] - q[1] * v[2]);
    const double tz = 2.0 * (q[1] * v[1] - q[2] * v[0]);
    o[0] = v[0] + q[0] * tx + (q[2] * tz - q[3] * ty);
    o[1] = v[1] + q[0] * ty + (q[3] * tx - q[1] * tz);
    o[2] = v[2] + q[0] * tz + (q[1] * ty - q[2] * tx);
}
// conj(q) * v
SLB_DEV void quat_rotate_inv(const double q[4], const double v[3], double o[3]) {
    const double qc[4] = {q[0], -q[1], -q[2], -q[3]};
    quat_rotate(qc, v, o);
}

// ---- compound manifold ops on register arrays -------------------------------------------------------
// y = x [+] (sign * d)
template <class L>
SLB_DEV void boxplus(const double *x, const double *d, double sign, double *y) {
#pragma unroll
    for (int b = 0; b < L::NB; ++b) {
        const int o = L::qoff(b);
        if (L::so3(b)) {
            const double v[3] = {sign * d[3 * b], sign * d[3 * b + 1], sign * d[3 * b + 2]};
            double e[4];
            so3_exp(v, 1.0, e);
            quat_mul(x + o, e, y + o);
        } else {
#pragma unroll
            for (int i = 0; i < 3; ++i) y[o + i] = x[o + i] + sign * d[3 * b + i];
        }
    }
}
// d = a [-] b
template <class L>
SLB_DEV void boxminus(const double *a, const double *b_, double *d) {
#pragma unroll
    for (int b = 0; b < L::NB; ++b) {
        const int o = L::qoff(b);
        if (L::so3(b)) {
            double r[4];
            quat_cmul(b_ + o, a + o, r);
            so3_log(r, d + 3 * b);
        } else {
#pragma unroll
            for (int i = 0; i < 3; ++i) d[3 * b + i] = a[o + i] - b_[o + i];
        }
    }
}

// ---- in-register packed Cholesky (lower, row-major packed).  Returns false on pivot <= 0. ----------
template <int N>
SLB_DEV bool chol_packed(double *A) {
    bool ok = true;
#pragma unroll
    for (int k = 0; k < N; ++k) {
        double x = A[tri(k, k)];
#pragma unroll
        for (int p = 0; p < k; ++p) x -= A[tri(k, p)] * A[tri(k, p)];
        ok = ok && (x > 0.0);
        x = sqrt(x);
        A[tri(k, k)] = x;
        const double inv = 1.0 / x;
#pragma unroll
        for (int i = k + 1; i < N; ++i) {
            double s = A[tri(i, k)];
#pragma unroll
            for (int p = 0; p < k; ++p) s -= A[tri(i, p)] * A[tri(k, p)];
            A[tri(i, k)] = s * inv;
        }
    }
    return ok;
}

// symmetric 3x3 inverse from packed lower S (s00 s10 s11 s20 s21 s22) -> packed lower
SLB_DEV void sym3_inverse(const double *S, double *Si) {
    const double a = S[0], b = S[1], c = S[2], d = S[3], e = S[4], f = S[5];
    const double c00 = c * f - e * e, c10 = d * e - b * f, c20 = b * e - c * d;
    const double det = a * c00 + b * c10 + d * c20;
    const double id = 1.0 / det;
    Si[0] = c00 * id;
    Si[1] = c10 * id;
    Si[2] = (a * f - d * d) * id;
    Si[3] = c20 * id;
    Si[4] = (b * d - a * e) * id;
    Si[5] = (a * c - b * b) * id;
}

SLB_DEV bool chi2_accept(double m2, int dof) {
    // 5% table, Usckf.hpp:794-855; dof 0 = accept_any_mahalanobis_distance; other dof reject.
    // (select chain, not an indexed array: a runtime-indexed table would live in local memory)
    if (dof == 0) return true;
    const double th = dof == 1 ? 3.84 : dof == 2 ? 5.99 : dof == 3 ? 7.81 : dof == 4 ? 9.49 : dof == 5 ? 11.07
                    : dof == 6 ? 12.59 : dof == 7 ? 14.07 : dof == 8 ? 15.51 : dof == 9 ? 16.92 : -1.0;
    return m2 < th;
}

}  // namespace slbd
