// slb_fusion.cu -- localization::DataModel<double,D>::fusion / operator+ / operator- over n
// independent pairs (DataModel.hpp:48-60,132-152).  Compiled with -fmad=false.
//
// The fusion is HBM-bound (d=6: 1008 B of dense instance-major traffic per pair against ~1.4 kflop),
// so the kernel spends its spare FP64 issue slots on following the reference's *as written*
// sequence -- inverse(C1), inverse(C2), inverse(sum), two mat-vecs, one mat-vec -- operation by
// operation in the order the CPU oracle uses (Eigen's fixed-size inverse: cofactors for D<=3,
// partial-pivot LU for D>3), without FMA contraction.  Division and sqrt are IEEE-exact on the
// device, so the results are bit-identical to the oracle's even on the cond~1e7 covariances of
// BASELINE config 5, where any reordering moves the answer by ~cond*eps.
//
// Data movement: a warp owns 32 consecutive pairs.  Their C matrices (32*D*D contiguous doubles)
// are copied global->shared with fully coalesced 16-byte loads into rows padded to an odd stride,
// each lane then owns one padded row (conflict-free), computes in registers, and the result goes
// back through the same staging so stores are coalesced too.
#include "slb_internal.h"
#include "slb_math.cuh"
#include "slb_ptx.cuh"

namespace slbd {

// IEEE-rounded a / d from r = RN(1/d): q0 = RN(a r), exact remainder by FMA, one correction (Markstein:
// with a correctly rounded reciprocal the corrected quotient is the correctly rounded a/d for normal,
// non-overflowing operands -- the same final step div.rn.f64 itself performs).  An LU inverse divides by
// each pivot 2D-1-k times, so the reciprocal (the expensive part of a division) is computed once per pivot.
SLB_DEV double div_by(double a, double d, double r) {
    const double q = __dmul_rn(a, r);
    const double rem = __fma_rn(-d, q, a);
    return __fma_rn(rem, r, q);
}

// Eigen PartialPivLU inverse restated (oracle/slo_core.hpp inverse_lu_fma): same pivot choice, same operation
// order, the multiply-subtract steps of the elimination and of both triangular solves fused (explicit __fma_rn here,
// std::fma there -- what Eigen's pmadd does in an FMA build of the reference), everything else unfused (-fmad=false),
// so the result is bit-identical to the CPU oracle.  Rows are
// swapped with predicated moves so LU stays in registers; each finished column of the inverse is handed
// to `sink(col, x)` instead of being kept (the caller stores or accumulates it), which keeps the live
// state at LU + two D-vectors.
template <int D, class Sink>
SLB_DEV void inverse_lu_cols(double *LU, Sink sink) {
    int perm[D];
    double rd[D];  // RN(1 / U_kk)
#pragma unroll
    for (int i = 0; i < D; ++i) perm[i] = i;
#pragma unroll
    for (int k = 0; k < D; ++k) {
        int piv = k;
        double best = fabs(LU[k * D + k]);
#pragma unroll
        for (int i = 0; i < D; ++i) {
            if (i > k) {
                const double v = fabs(LU[i * D + k]);
                if (v > best) { best = v; piv = i; }
            }
        }
#pragma unroll
        for (int i = 0; i < D; ++i) {
            if (i > k) {
                const bool sw = piv == i;
#pragma unroll
                for (int j = 0; j < D; ++j) {
                    const double t = LU[k * D + j], u = LU[i * D + j];
                    LU[k * D + j] = sw ? u : t;
                    LU[i * D + j] = sw ? t : u;
                }
                const int tp = perm[k], up = perm[i];
                perm[k] = sw ? up : tp;
                perm[i] = sw ? tp : up;
            }
        }
        const double d = LU[k * D + k];
        const double r = __drcp_rn(d);
        rd[k] = r;
#pragma unroll
        for (int i = 0; i < D; ++i)
            if (i > k) LU[i * D + k] = div_by(LU[i * D + k], d, r);
#pragma unroll
        for (int i = 0; i < D; ++i) {
            if (i > k) {
                const double lik = LU[i * D + k];
#pragma unroll
                for (int j = 0; j < D; ++j)
                    if (j > k) LU[i * D + j] = __fma_rn(-lik, LU[k * D + j], LU[i * D + j]);
            }
        }
    }
    // one column at a time (rolled): the six solves unrolled side by side need > 200 registers, and the
    // kernel is HBM-bound, so the shorter schedule buys nothing
#pragma unroll 1
    for (int col = 0; col < D; ++col) {
        double y[D], x[D];
#pragma unroll
        for (int i = 0; i < D; ++i) {
            double s = (perm[i] == col) ? 1.0 : 0.0;
#pragma unroll
            for (int p = 0; p < D; ++p)
                if (p < i) s = __fma_rn(-LU[i * D + p], y[p], s);
            y[i] = s;
        }
#pragma unroll
        for (int i = D - 1; i >= 0; --i) {
            double s = y[i];
#pragma unroll
            for (int p = 0; p < D; ++p)
                if (p > i) s = __fma_rn(-LU[i * D + p], x[p], s);
            x[i] = div_by(s, LU[i * D + i], rd[i]);
        }
        sink(col, x);
    }
}

// Eigen fixed 3x3 inverse (cofactors / determinant), oracle/slo_core.hpp inverse_3x3_cofactor.
SLB_DEV void inverse_3x3(const double *A, double *C) {
#define SLB_COF(i, j) \
    (A[((i + 1) % 3) * 3 + (j + 1) % 3] * A[((i + 2) % 3) * 3 + (j + 2) % 3] - A[((i + 1) % 3) * 3 + (j + 2) % 3] * A[((i + 2) % 3) * 3 + (j + 1) % 3])
    const double c00 = SLB_COF(0, 0), c10 = SLB_COF(1, 0), c20 = SLB_COF(2, 0);
    const double det = c00 * A[0] + c10 * A[3] + c20 * A[6];
    const double invdet = 1.0 / det;
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j) C[j * 3 + i] = SLB_COF(i, j) * invdet;
#undef SLB_COF
}

// v[col] for a runtime col without indexing the register array (that would spill it to local memory)
template <int D>
SLB_DEV double pick(const double *v, int col) {
    double r = v[0];
#pragma unroll
    for (int i = 1; i < D; ++i) r = (col == i) ? v[i] : r;
    return r;
}

// inverse of the DxD matrix held row-major in registers A (destroyed for D > 3); columns go to sink
template <int D, class Sink>
SLB_DEV void inverse_fixed_cols(double *A, Sink sink) {
    if (D == 3) {
        double X[9];
        inverse_3x3(A, X);
#pragma unroll
        for (int col = 0; col < 3; ++col) {
            const double x[3] = {X[col], X[3 + col], X[6 + col]};
            sink(col, x);
        }
    } else {
        inverse_lu_cols<D>(A, sink);
    }
}

constexpr int FUSE_WARPS = 4;

template <int D>
struct FuseCfg {
    static constexpr int DD = D * D;
    static constexpr int RS = (DD % 2 == 0) ? DD + 1 : DD;  // odd row stride: conflict-free per-lane rows
    static constexpr size_t SMEM = (size_t)FUSE_WARPS * 2 * 32 * RS * sizeof(double);
};

// OP: 0 fusion, +1 operator+, -1 operator-
template <int D, int OP>
__global__ void __launch_bounds__(FUSE_WARPS * 32) datamodel_kernel(int64_t n, const double *x1,  // xo / Co may alias x1 / C1 (in-place fusion): no restrict
                                                                  const double *C1,
                                                                  const double *__restrict__ x2,
                                                                  const double *__restrict__ C2, double *xo,
                                                                  double *Co) {
    constexpr int DD = FuseCfg<D>::DD, RS = FuseCfg<D>::RS;
    extern __shared__ double sbuf[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    double *s1 = sbuf + (size_t)warp * 2 * 32 * RS, *s2 = s1 + 32 * RS;
    const int64_t nwarps_total = (int64_t)gridDim.x * FUSE_WARPS;
    for (int64_t tile = (int64_t)blockIdx.x * FUSE_WARPS + warp; tile * 32 < n; tile += nwarps_total) {
        const int64_t base = tile * 32;
        const int cnt = (int)((n - base) < 32 ? (n - base) : 32);
        // coalesced asynchronous stage-in of the two covariance tiles (LDGSTS, 8 B per lane)
        const double *g1 = C1 + base * DD, *g2 = C2 + base * DD;
        if (cnt == 32) {
#pragma unroll
            for (int it = 0; it < DD; ++it) {
                const int e = it * 32 + lane;
                const int r = e / DD, c = e - r * DD;
                cp_async8(s1 + r * RS + c, g1 + e);
                cp_async8(s2 + r * RS + c, g2 + e);
            }
        } else {
            for (int e = lane; e < cnt * DD; e += 32) {
                const int r = e / DD, c = e - r * DD;
                cp_async8(s1 + r * RS + c, g1 + e);
                cp_async8(s2 + r * RS + c, g2 + e);
            }
        }
        double a[D], b[D], xr[D];
        const bool act = lane < cnt;
        if (act) {
#pragma unroll
            for (int e = 0; e < D; ++e) a[e] = x1[(base + lane) * D + e];
            if (OP != 0) {
#pragma unroll
                for (int e = 0; e < D; ++e) b[e] = x2[(base + lane) * D + e];
            }
        }
        cp_async_wait_all();
        __syncwarp();
        double *r1 = s1 + lane * RS, *r2 = s2 + lane * RS;  // this lane's padded rows
        if (act) {
            if (OP == 0) {
                // fusion (DataModel.hpp:48-60) in the oracle's order: I1 = C1^-1, I2 = C2^-1, P = (I1 + I2)^-1,
                // x = P (I1 x1 + I2 x2).  The mat-vecs accumulate column by column as the inverses are produced
                // (the same left-to-right sums as a row-wise mat-vec), I1 and I1 + I2 are parked in the row of C1.
                double M[DD], ya[D], yb[D];
#pragma unroll
                for (int e = 0; e < DD; ++e) M[e] = r1[e];
#pragma unroll
                for (int i = 0; i < D; ++i) ya[i] = 0.0;
                inverse_fixed_cols<D>(M, [&](int col, const double *x) {
                    const double ac = pick<D>(a, col);
#pragma unroll
                    for (int i = 0; i < D; ++i) {
                        r1[i * D + col] = x[i];
                        ya[i] = ya[i] + x[i] * ac;
                    }
                });
#pragma unroll
                for (int e = 0; e < DD; ++e) M[e] = r2[e];
#pragma unroll
                for (int i = 0; i < D; ++i) {  // x2 is fetched only now: fewer live registers during inverse 1
                    yb[i] = 0.0;
                    b[i] = x2[(base + lane) * D + i];
                }
                inverse_fixed_cols<D>(M, [&](int col, const double *x) {
                    const double bc = pick<D>(b, col);
#pragma unroll
                    for (int i = 0; i < D; ++i) {
                        r1[i * D + col] = r1[i * D + col] + x[i];
                        yb[i] = yb[i] + x[i] * bc;
                    }
                });
#pragma unroll
                for (int e = 0; e < DD; ++e) M[e] = r1[e];
#pragma unroll
                for (int i = 0; i < D; ++i) { ya[i] = ya[i] + yb[i]; xr[i] = 0.0; }
                inverse_fixed_cols<D>(M, [&](int col, const double *x) {
                    const double yc = pick<D>(ya, col);
#pragma unroll
                    for (int i = 0; i < D; ++i) {
                        r1[i * D + col] = x[i];
                        xr[i] = xr[i] + x[i] * yc;
                    }
                });
            } else {
#pragma unroll
                for (int e = 0; e < DD; ++e) r1[e] = r1[e] + r2[e];  // operator- ALSO adds (:149)
#pragma unroll
                for (int e = 0; e < D; ++e) xr[e] = OP > 0 ? a[e] + b[e] : a[e] - b[e];
            }
        }
        if (act) {
#pragma unroll
            for (int e = 0; e < D; ++e) xo[(base + lane) * D + e] = xr[e];
        }
        __syncwarp();
        double *go = Co + base * DD;
        if (cnt == 32) {
#pragma unroll
            for (int it = 0; it < DD; ++it) {
                const int e = it * 32 + lane;
                const int r = e / DD, c = e - r * DD;
                go[e] = s1[r * RS + c];
            }
        } else {
            for (int e = lane; e < cnt * DD; e += 32) {
                const int r = e / DD, c = e - r * DD;
                go[e] = s1[r * RS + c];
            }
        }
        __syncwarp();
    }
}

}  // namespace slbd

namespace slb {

template <int D, int OP>
static int launch_dm(int64_t n, const double *x1, const double *C1, const double *x2, const double *C2,
                     double *xo, double *Co, cudaStream_t s) {
    const int64_t tiles = (n + 31) / 32;
    int64_t blocks = (tiles + slbd::FUSE_WARPS - 1) / slbd::FUSE_WARPS;
    const int64_t cap = (int64_t)sm_count() * 16;  // persistent: a multiple of the SM count
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    return launch(slbd::datamodel_kernel<D, OP>, (int)blocks, slbd::FUSE_WARPS * 32, slbd::FuseCfg<D>::SMEM, s, n, x1, C1, x2,
                  C2, xo, Co);
}

int launch_fusion(int d, int64_t n, int op, const double *x1, const double *C1, const double *x2,
                  const double *C2, double *xo, double *Co, cudaStream_t s) {
    if (n <= 0) return SLB_OK;
#define SLB_DM(D_)                                                                 \
    if (d == D_) {                                                                 \
        if (op == 0) return launch_dm<D_, 0>(n, x1, C1, x2, C2, xo, Co, s);        \
        if (op > 0) return launch_dm<D_, 1>(n, x1, C1, x2, C2, xo, Co, s);         \
        return launch_dm<D_, -1>(n, x1, C1, x2, C2, xo, Co, s);                    \
    }
    SLB_DM(3)
    SLB_DM(6)
#undef SLB_DM
    return set_error(SLB_ERR_INVALID, "datamodel: only d = 3 and d = 6 are built");
}

}  // namespace slb
