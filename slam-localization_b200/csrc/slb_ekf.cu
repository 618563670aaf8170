// slb_ekf.cu -- SURVEY 8(f) row f2: the error-state EKF of src/filters/UsckfError.hpp, one instance per WARP.
//
//   ekfPredict(F, Q)          UsckfError.hpp:87-137   ->  ekf_predict_kernel
//   ekfUpdate(z, H, R, mt)    UsckfError.hpp:322-384  ->  ekf_update_kernel<M>        (Joseph form + symmetrisation)
//   ekfSingleUpdate(z,H,R,mt) UsckfError.hpp:489-571  ->  ekf_single_update_kernel<M> (Joseph form on the statek_i block)
//   cloning()                 UsckfError.hpp:573-603  ->  ekf_clone_kernel
//
// Data in HBM is what the reference object holds, instance-major: mu_state as 3 x 16 q-vector scalars
// (pos vel quat(w,x,y,z) gbias abias per single state -- the 15-DOF layout of :527-531; the reference's own type
// is not in its tree), mu_error vectorised (45), Pk_error as a DENSE 45 x 45 row-major matrix.  Only the lower
// triangle of a covariance block is read (like every other kernel here); both triangles are written.
//
// All three filter kernels are HBM-bound (2-3 flop/B): a warp streams its instance's rows with coalesced
// loads into shared memory, does the O(N^2 m) algebra there and streams the result back.
// The Joseph form (I-KH) P (I-KH)^T + K R K^T is evaluated in its expanded, algebraically identical form
//   P - K A^T - A K^T + K S K^T,   A = P H^T,  S = H A + R
// (O(N^2 m) instead of two N^3 products) and symmetrised as 0.5 (P + P^T) like :359.
#include "slb_internal.h"
#include "slb_math.cuh"
#include "slb_ptx.cuh"

namespace slbd {

constexpr int EKF_NS = 15, EKF_NA = 45, EKF_QS = 16, EKF_QA = 48;

// closed-form inverse of a general 3x3 (Eigen's fixed-size path: cofactors / determinant)
SLB_DEV void inv3(const double *A, double *C) {
    auto a = [&](int i, int j) { return A[i * 3 + j]; };
    auto cof = [&](int i, int j) {
        const int i1 = (i + 1) % 3, i2 = (i + 2) % 3, j1 = (j + 1) % 3, j2 = (j + 2) % 3;
        return a(i1, j1) * a(i2, j2) - a(i1, j2) * a(i2, j1);
    };
    const double c00 = cof(0, 0), c10 = cof(1, 0), c20 = cof(2, 0);
    const double det = c00 * a(0, 0) + c10 * a(1, 0) + c20 * a(2, 0);
    const double id = 1.0 / det;
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j) C[j * 3 + i] = cof(i, j) * id;
}

// ---- ekfPredict ---------------------------------------------------------------------------------------
// block row i = rows 30..44:  [P_ik P_il P_ii] <- F [P_ik P_il P_ii],  P_ii <- (F P_ii) F^T + Q,  columns 30..44 of
// rows 0..29 by symmetry (the reference updates P_ki = P_ki F^T separately, :109-116: the same numbers for a
// symmetric Pk_error).  Both products are 8x8x4 FP64 DMMA tiles fed from shared memory: Y = F * [block row] is
// column-wise independent, so each 8-column strip is computed into registers and written back in place.
constexpr int EKP_FS = 20, EKP_RS = 52;   // row strides of F (16 x 16 padded) and of the block row (16 x 48 padded):
                                          // = 4 (mod 16) doubles, so a 4 x 8 fragment load touches 32 distinct banks
constexpr int EKP_SM = 16 * EKP_FS + 16 * EKP_RS;
template <int WPB>
__global__ void __launch_bounds__(WPB * 32) ekf_predict_kernel(int64_t n, double *err, double *P, const double *F, const double *Q) {
    extern __shared__ __align__(16) double sm[];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int64_t inst = (int64_t)blockIdx.x * WPB + w;
    if (inst >= n) return;
    const int fr = lane >> 2, fk = lane & 3;   // DMMA fragment coordinates
    double *Fs = sm + (size_t)w * EKP_SM, *Rs = Fs + 16 * EKP_FS;
    double *Pg = P + inst * (EKF_NA * EKF_NA);
    const double *Fg = F + inst * (EKF_NS * EKF_NS);
    // 8-byte LDGSTS: the loads of a record are all issued before the first one lands (instance records are only 8-byte
    // aligned -- 2025 doubles -- so the 16-byte form does not apply); one wait for the lot.
    for (int e = lane; e < 225; e += 32) cp_async8(Fs + (e / 15) * EKP_FS + e % 15, Fg + e);
    for (int e = lane; e < 675; e += 32) cp_async8(Rs + (e / 45) * EKP_RS + e % 45, Pg + 30 * 45 + e);
    // zero padding of the k-dimension (column 15 of F, row 15 of the block row) and of the unused columns 45..47
    if (lane < 16) { Fs[lane * EKP_FS + 15] = 0.0; Fs[15 * EKP_FS + lane] = 0.0; }
    for (int e = lane; e < 48; e += 32) Rs[15 * EKP_RS + e] = 0.0;
    for (int e = lane; e < 48; e += 32) Rs[(e / 3) * EKP_RS + 45 + e % 3] = 0.0;
    double ei = lane < 15 ? err[inst * EKF_NA + 30 + lane] : 0.0;
    cp_async_wait_all();
    __syncwarp();
    // mu_error.statek_i <- F mu_error.statek_i (:93)
    {
        double s = 0.0;
#pragma unroll
        for (int k = 0; k < 15; ++k) {
            const double ek = __shfl_sync(FULL, ei, k);
            if (lane < 15) s += Fs[lane * EKP_FS + k] * ek;
        }
        if (lane < 15) err[inst * EKF_NA + 30 + lane] = s;
    }
    // A fragments of F: A[m][k] = F[8I + fr][k0 + fk]
    double fa[2][4];
#pragma unroll
    for (int I = 0; I < 2; ++I)
#pragma unroll
        for (int kq = 0; kq < 4; ++kq) fa[I][kq] = Fs[(8 * I + fr) * EKP_FS + 4 * kq + fk];
    // Y = F * block row, strip by strip (8 columns), in place
#pragma unroll 2
    for (int J = 0; J < 6; ++J) {
        double y0[2] = {0.0, 0.0}, y1[2] = {0.0, 0.0};
#pragma unroll
        for (int kq = 0; kq < 4; ++kq) {
            const double bv = Rs[(4 * kq + fk) * EKP_RS + 8 * J + fr];   // B[k][n] = row k, column 8J + n
            dmma884(y0[0], y0[1], fa[0][kq], bv);
            dmma884(y1[0], y1[1], fa[1][kq], bv);
        }
        __syncwarp();
        Rs[fr * EKP_RS + 8 * J + 2 * fk] = y0[0];
        Rs[fr * EKP_RS + 8 * J + 2 * fk + 1] = y0[1];
        Rs[(8 + fr) * EKP_RS + 8 * J + 2 * fk] = y1[0];
        Rs[(8 + fr) * EKP_RS + 8 * J + 2 * fk + 1] = y1[1];
    }
    __syncwarp();
    // P_ii = Y_ii F^T + Q (:96): A = Y[:, 30 + k], B[k][n] = F[n][k] (the A-fragment pattern of F)
    {
        double c[2][2][2];
#pragma unroll
        for (int I = 0; I < 2; ++I)
#pragma unroll
            for (int J = 0; J < 2; ++J) c[I][J][0] = c[I][J][1] = 0.0;
#pragma unroll
        for (int kq = 0; kq < 4; ++kq) {
            const double a0 = Rs[fr * EKP_RS + 30 + 4 * kq + fk], a1 = Rs[(8 + fr) * EKP_RS + 30 + 4 * kq + fk];
            dmma884(c[0][0][0], c[0][0][1], a0, fa[0][kq]);
            dmma884(c[0][1][0], c[0][1][1], a0, fa[1][kq]);
            dmma884(c[1][0][0], c[1][0][1], a1, fa[0][kq]);
            dmma884(c[1][1][0], c[1][1][1], a1, fa[1][kq]);
        }
        __syncwarp();
#pragma unroll
        for (int I = 0; I < 2; ++I)
#pragma unroll
            for (int J = 0; J < 2; ++J)
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    const int r = 8 * I + fr, cc = 8 * J + 2 * fk + h;
                    if (r < 15 && cc < 15) Rs[r * EKP_RS + 30 + cc] = c[I][J][h] + __ldg(Q + r * 15 + cc);
                }
    }
    __syncwarp();
    for (int e = lane; e < 675; e += 32) Pg[30 * 45 + e] = Rs[(e / 45) * EKP_RS + e % 45];
    // mirrored blocks: row k < 30, columns 30..44
    for (int e = lane; e < 450; e += 32) {
        const int k = e / 15, c = e - k * 15;
        Pg[k * 45 + 30 + c] = Rs[c * EKP_RS + k];
    }
}

// ---- ekfUpdate: N = 45 on the whole Pk_error, M = 3 ---------------------------------------------------------
// shared memory per warp: packed lower triangle (also the result), A | K | G rows, H
template <int N, int M>
struct EkuCfg {
    static constexpr int NP = N * (N + 1) / 2;
    static constexpr int ROW = 12;  // K(3) A(3) G(3) + pad: 16-byte aligned rows
    static constexpr int RO = (NP + 1) / 2 * 2;  // offset of the rows (even: 16-byte aligned for the vector loads)
    static constexpr int SM = (RO + N * ROW + M * N + 1) / 2 * 2;
};

// Joseph-form update of the packed lower triangle Pl (N x N) held in shared memory; H (M x N) in shared memory.
// Returns the acceptance decision; innovation in `innov`.
template <int N, int M>
SLB_DEV bool joseph_update(double *Pl, double *rows, const double *Hs, const double *xhat /* smem, N */, const double *zg,
                           const double *Rg, int gate, int lane, double *innov) {
    typedef EkuCfg<N, M> C;
    static_assert(M == 3, "S^-1 is the closed-form 3x3 inverse");
    static_assert(N <= 64, "two rows per lane");
    // A = P H^T as 8x8x4 FP64 DMMA tiles: M-dim = rows of P, K-dim = columns j (padded to a multiple of 4, H = 0
    // there), N-dim = measurement index (3 of 8 columns used).  P is symmetric packed: entry (i,j) = Pl[tri(max,min)].
    const int i0 = lane, i1 = lane + 32;
    {
        const int fr = lane >> 2, fk = lane & 3;
        constexpr int NT = (N + 7) / 8, KQ = (N + 3) / 4;
        double hb[KQ];   // B[k = j][n = fr] = H[fr][j]
#pragma unroll
        for (int kq = 0; kq < KQ; ++kq) {
            const int j = 4 * kq + fk;
            hb[kq] = (fr < M && j < N) ? Hs[fr * N + j] : 0.0;
        }
#pragma unroll 1
        for (int I = 0; I < NT; ++I) {
            const int ri = min(8 * I + fr, N - 1), tr0 = tri(ri, 0);
            double d0 = 0.0, d1 = 0.0;
#pragma unroll
            for (int kq = 0; kq < KQ; ++kq) {
                const int jc = min(4 * kq + fk, N - 1);
                dmma884(d0, d1, Pl[ri >= jc ? tr0 + jc : tri(jc, ri)], hb[kq]);
            }
            const int r = 8 * I + fr;
            if (r < N) {
                if (fk == 0) { rows[r * C::ROW + 3] = d0; rows[r * C::ROW + 4] = d1; }
                if (fk == 1) rows[r * C::ROW + 5] = d0;
            }
        }
    }
    __syncwarp();
    double A0[M], A1[M];
#pragma unroll
    for (int c = 0; c < M; ++c) {
        A0[c] = i0 < N ? rows[i0 * C::ROW + 3 + c] : 0.0;
        A1[c] = i1 < N ? rows[i1 * C::ROW + 3 + c] : 0.0;
    }
    __syncwarp();
    // S = H A + R and H x_hat: each lane adds the terms of its own rows, one butterfly reduction for the 12 sums
    double S[M * M], hx[M];
#pragma unroll
    for (int r = 0; r < M; ++r) {
        const double h0 = i0 < N ? Hs[r * N + i0] : 0.0, h1 = i1 < N ? Hs[r * N + i1] : 0.0;
        double t = fma(h0, i0 < N ? xhat[i0] : 0.0, h1 * (i1 < N ? xhat[i1] : 0.0));
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(FULL, t, o);
        hx[r] = t;
#pragma unroll
        for (int c = 0; c < M; ++c) {
            double v = fma(h0, A0[c], h1 * A1[c]);
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(FULL, v, o);
            S[r * M + c] = v + __ldg(Rg + r * M + c);
        }
    }
    double Si[M * M];
    inv3(S, Si);
    double m2 = 0.0;
#pragma unroll
    for (int r = 0; r < M; ++r) innov[r] = zg[r] - hx[r];
#pragma unroll
    for (int r = 0; r < M; ++r) {
        double t = 0.0;
#pragma unroll
        for (int c = 0; c < M; ++c) t += Si[r * M + c] * innov[c];
        m2 += innov[r] * t;
    }
    const bool accept = chi2_accept(m2, gate == 0 ? 0 : M - 1);  // dof = innovation.size() - 1 (:350)
    // K = A S^-1, G = K S - A
    auto finish = [&](const double *Ar, int i) {
        double K[M];
#pragma unroll
        for (int c = 0; c < M; ++c) {
            double s = 0.0;
#pragma unroll
            for (int p = 0; p < M; ++p) s += Ar[p] * Si[p * M + c];
            K[c] = s;
        }
#pragma unroll
        for (int c = 0; c < M; ++c) {
            double s = -Ar[c];
#pragma unroll
            for (int p = 0; p < M; ++p) s = fma(K[p], S[p * M + c], s);
            rows[i * C::ROW + c] = K[c];
            rows[i * C::ROW + 6 + c] = s;
        }
    };
    if (i0 < N) finish(A0, i0);
    if (i1 < N) finish(A1, i1);
    __syncwarp();
    if (!accept) return false;
    // P'_ij = P_ij - 0.5 (K_i.A_j + A_i.K_j) + 0.5 (G_i.K_j + K_i.G_j) = P_ij + X_i . Y_j with the 12-vectors
    // X = [-K/2 | -A/2 | G/2 | K/2], Y = [A | K | K | G]: a rank-12 update of the lower 8x8 tiles as FP64 DMMA,
    // fragments picked straight out of the K | A | G rows (rows beyond N only feed accumulator entries that are dropped).
    {
        const int fr = lane >> 2, fk = lane & 3;
        int xo[3], yo[3];
        double xs[3];
#pragma unroll
        for (int kq = 0; kq < 3; ++kq) {
            const int k = 4 * kq + fk;
            xo[kq] = k < 9 ? k : k - 9;
            xs[kq] = k < 6 ? -0.5 : 0.5;
            yo[kq] = k < 3 ? 3 + k : (k < 6 ? k - 3 : (k < 9 ? k - 6 : k - 3));
        }
        constexpr int NT = (N + 7) / 8;
#pragma unroll 1
        for (int I = 0; I < NT; ++I) {
            const double *ri = rows + min(8 * I + fr, N - 1) * C::ROW;
            const double xa0 = ri[xo[0]] * xs[0], xa1 = ri[xo[1]] * xs[1], xa2 = ri[xo[2]] * xs[2];
            const int r = 8 * I + fr;
#pragma unroll 1
            for (int J = 0; J <= I; ++J) {
                const double *rj = rows + min(8 * J + fr, N - 1) * C::ROW;
                double d0 = 0.0, d1 = 0.0;
                dmma884(d0, d1, xa0, rj[yo[0]]);
                dmma884(d0, d1, xa1, rj[yo[1]]);
                dmma884(d0, d1, xa2, rj[yo[2]]);
                const int c = 8 * J + 2 * fk;
                if (r < N) {
                    double *pr = Pl + tri(r, 0);
                    if (c <= r) pr[c] += d0;
                    if (c + 1 <= r) pr[c + 1] += d1;
                }
            }
        }
    }
    __syncwarp();
    return true;
}

template <int M, int WPB>
__global__ void __launch_bounds__(WPB * 32) ekf_update_kernel(int64_t n, const double *mu, double *P, const double *z, const double *H,
                                                              const double *R, int gate, double *ret, int32_t *accepted) {
    constexpr int N = EKF_NA;
    typedef EkuCfg<N, M> C;
    extern __shared__ __align__(16) double sm[];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int64_t inst = (int64_t)blockIdx.x * WPB + w;
    if (inst >= n) return;
    double *Pl = sm + (size_t)w * (C::SM + N + 1) , *rows = Pl + C::RO, *Hs = rows + N * C::ROW, *xh = sm + (size_t)w * (C::SM + N + 1) + C::SM;
    double *Pg = P + inst * (N * N);
    // lower triangle of the dense matrix -> packed rows: one flat loop over the packed index (a nested row / column loop
    // diverges on every row and spent 2 300 instructions per warp issuing 33 copies per lane)
    for (int e = lane; e < C::NP; e += 32) {
        int i = (int)((sqrtf(8.0f * e + 1.0f) - 1.0f) * 0.5f);
        i += (tri(i + 1, 0) <= e) - (tri(i, 0) > e);
        cp_async8(Pl + e, Pg + i * N + (e - tri(i, 0)));
    }
    for (int e = lane; e < M * N; e += 32) Hs[e] = __ldg(H + e);
    // x_hat = mu_state vectorised with the error-quaternion convention (:331)
    for (int e = lane; e < N; e += 32) {
        const int s = e / EKF_NS, c = e - s * EKF_NS;
        xh[e] = mu[inst * EKF_QA + s * EKF_QS + (c < 6 ? c : c + 1)];
    }
    cp_async_wait_all();
    __syncwarp();
    double innov[M];
    const bool ok = joseph_update<N, M>(Pl, rows, Hs, xh, z + inst * M, R, gate, lane, innov);
    if (lane == 0) {
        accepted[inst] = ok ? 1 : 0;
#pragma unroll
        for (int c = 0; c < M; ++c) ret[inst * M + c] = ok ? 0.0 : innov[c];  // :361 / :371
    }
    if (!ok) return;
    {   // dense rows out, coalesced; (i, j) advance incrementally instead of a division per element
        int i = 0, j = lane;
        for (int e = lane; e < N * N; e += 32) {
            Pg[e] = Pl[i >= j ? tri(i, j) : tri(j, i)];
            j += 32;
            if (j >= N) { j -= N; ++i; }
        }
    }
}

// ---- ekfSingleUpdate: the 15 x 15 statek_i block and mu_state.statek_i --------------------------------------
template <int M, int WPB>
__global__ void __launch_bounds__(WPB * 32) ekf_single_update_kernel(int64_t n, double *mu, const double *err, double *P, const double *z,
                                                                     const double *H, const double *R, int gate, int32_t *accepted) {
    constexpr int N = EKF_NS;
    typedef EkuCfg<N, M> C;
    extern __shared__ __align__(16) double sm[];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int64_t inst = (int64_t)blockIdx.x * WPB + w;
    if (inst >= n) return;
    double *Pl = sm + (size_t)w * (C::SM + N + 1), *rows = Pl + C::RO, *Hs = rows + N * C::ROW, *xk = sm + (size_t)w * (C::SM + N + 1) + C::SM;
    double *Pg = P + inst * (EKF_NA * EKF_NA);
    for (int e = lane; e < N * N; e += 32) {
        const int i = e / N, j = e - i * N;
        if (j <= i) cp_async8(Pl + tri(i, j), Pg + (30 + i) * EKF_NA + 30 + j);
    }
    for (int e = lane; e < M * N; e += 32) Hs[e] = __ldg(H + e);
    if (lane < N) xk[lane] = err[inst * EKF_NA + 30 + lane];
    cp_async_wait_all();
    __syncwarp();
    double innov[M];
    const bool ok = joseph_update<N, M>(Pl, rows, Hs, xk, z + inst * M, R, gate, lane, innov);
    if (lane == 0) accepted[inst] = ok ? 1 : 0;
    if (ok) {
        for (int e = lane; e < N * N; e += 32) {
            const int i = e / N, j = e - i * N;
            Pg[(30 + i) * EKF_NA + 30 + j] = Pl[i >= j ? tri(i, j) : tri(j, i)];
        }
    }
    // corrections (:553-568), applied whether or not the gate accepted; x = xk (+ K innovation when accepted)
    double x = 0.0;
    if (lane < N) {
        x = xk[lane];
        if (ok) {
#pragma unroll
            for (int c = 0; c < M; ++c) x = fma(rows[lane * C::ROW + c], innov[c], x);
        }
    }
    double *s = mu + inst * EKF_QA + 2 * EKF_QS;
    const double qx = __shfl_sync(FULL, x, 6), qy = __shfl_sync(FULL, x, 7), qz = __shfl_sync(FULL, x, 8);
    if (lane < 6) s[lane] += x;                       // pos, vel
    else if (lane >= 9 && lane < N) s[lane + 1] += x;  // gbias, abias
    if (lane == 6) {
        const double q0[4] = {s[6], s[7], s[8], s[9]}, qe[4] = {1.0, qx, qy, qz};
        double q[4];
        quat_mul(q0, qe, q);
        const double nn = sqrt(q[0] * q[0] + q[1] * q[1] + q[2] * q[2] + q[3] * q[3]);
#pragma unroll
        for (int c = 0; c < 4; ++c) s[6 + c] = q[c] / nn;
    }
}

// ---- cloning() (:573-603): every 15 x 15 block <- P_ii, statek = statek_l = statek_i ---------------------------
__global__ void ekf_clone_kernel(int64_t n, double *mu, double *err, double *P) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    constexpr int PER = EKF_NA * EKF_NA + 2 * EKF_QS + 2 * EKF_NS;
    if (t >= n * PER) return;
    const int64_t inst = t / PER;
    const int e = (int)(t - inst * PER);
    if (e < EKF_NA * EKF_NA) {
        const int i = e / EKF_NA, j = e - i * EKF_NA;
        if (i >= 30 && j >= 30) return;
        P[inst * (EKF_NA * EKF_NA) + e] = P[inst * (EKF_NA * EKF_NA) + (30 + i % 15) * EKF_NA + 30 + j % 15];
    } else if (e < EKF_NA * EKF_NA + 2 * EKF_QS) {
        const int c = e - EKF_NA * EKF_NA;
        mu[inst * EKF_QA + c] = mu[inst * EKF_QA + 2 * EKF_QS + c % EKF_QS];
    } else {
        const int c = e - EKF_NA * EKF_NA - 2 * EKF_QS;
        err[inst * EKF_NA + c] = err[inst * EKF_NA + 2 * EKF_NS + c % EKF_NS];
    }
}

}  // namespace slbd

using namespace slb;

extern "C" {

int slb_ekf_predict(int64_t n, double *err, double *P, const double *F, const double *Q, void *stream) {
    if (n < 0 || !err || !P || !F || !Q) return set_error(SLB_ERR_INVALID, "slb_ekf_predict: bad argument");
    if (n == 0) return SLB_OK;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        return set_error(SLB_ERR_NO_DEVICE, "slb_ekf_predict: no CUDA device (this engine has no CPU fallback)");
    }
    constexpr int WPB = 8;
    constexpr size_t smem = (size_t)WPB * slbd::EKP_SM * 8;
    auto kern = slbd::ekf_predict_kernel<WPB>;
    SLB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<(unsigned)((n + WPB - 1) / WPB), WPB * 32, smem, (cudaStream_t)stream>>>(n, err, P, F, Q);
    count_launch();
    SLB_CUDA(cudaGetLastError());
    return SLB_OK;
}

int slb_ekf_update(int64_t n, int m, const double *mu, double *P, const double *z, const double *H, const double *R, int gate,
                   double *ret, int32_t *accepted, void *stream) {
    if (n < 0 || !mu || !P || !z || !H || !R || !ret || !accepted) return set_error(SLB_ERR_INVALID, "slb_ekf_update: bad argument");
    if (m != 3) return set_error(SLB_ERR_INVALID, "slb_ekf_update: built for m = 3 (delay-position / velocity measurements)");
    if (n == 0) return SLB_OK;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        return set_error(SLB_ERR_NO_DEVICE, "slb_ekf_update: no CUDA device (this engine has no CPU fallback)");
    }
    constexpr int WPB = 8;
    constexpr size_t smem = (size_t)WPB * (slbd::EkuCfg<45, 3>::SM + 46) * 8;
    auto kern = slbd::ekf_update_kernel<3, WPB>;
    SLB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<(unsigned)((n + WPB - 1) / WPB), WPB * 32, smem, (cudaStream_t)stream>>>(n, mu, P, z, H, R, gate, ret, accepted);
    count_launch();
    SLB_CUDA(cudaGetLastError());
    return SLB_OK;
}

int slb_ekf_single_update(int64_t n, int m, double *mu, const double *err, double *P, const double *z, const double *H,
                          const double *R, int gate, int32_t *accepted, void *stream) {
    if (n < 0 || !mu || !err || !P || !z || !H || !R || !accepted) return set_error(SLB_ERR_INVALID, "slb_ekf_single_update: bad argument");
    if (m != 3) return set_error(SLB_ERR_INVALID, "slb_ekf_single_update: built for m = 3");
    if (n == 0) return SLB_OK;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        return set_error(SLB_ERR_NO_DEVICE, "slb_ekf_single_update: no CUDA device (this engine has no CPU fallback)");
    }
    constexpr int WPB = 8;
    constexpr size_t smem = (size_t)WPB * (slbd::EkuCfg<15, 3>::SM + 16) * 8;
    auto kern = slbd::ekf_single_update_kernel<3, WPB>;
    kern<<<(unsigned)((n + WPB - 1) / WPB), WPB * 32, smem, (cudaStream_t)stream>>>(n, mu, err, P, z, H, R, gate, accepted);
    count_launch();
    SLB_CUDA(cudaGetLastError());
    return SLB_OK;
}

int slb_ekf_clone(int64_t n, double *mu, double *err, double *P, void *stream) {
    if (n < 0 || !mu || !err || !P) return set_error(SLB_ERR_INVALID, "slb_ekf_clone: bad argument");
    if (n == 0) return SLB_OK;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        return set_error(SLB_ERR_NO_DEVICE, "slb_ekf_clone: no CUDA device (this engine has no CPU fallback)");
    }
    const int64_t work = n * (45 * 45 + 32 + 30);
    slbd::ekf_clone_kernel<<<(unsigned)((work + 255) / 256), 256, 0, (cudaStream_t)stream>>>(n, mu, err, P);
    count_launch();
    SLB_CUDA(cudaGetLastError());
    return SLB_OK;
}

}  // extern "C"
