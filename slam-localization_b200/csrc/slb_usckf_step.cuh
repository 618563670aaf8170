// slb_usckf_step.cuh -- localization::Usckf predict (Usckf.hpp:107-244) and update (:246-308) of one filter
// instance per WARP with the instance record RESIDENT IN SHARED MEMORY: one TMA bulk load brings the lower triangle
// of Pk (tiled, prec) and the mean in, predict and update work on it in place, one TMA bulk store writes it back, so a
// fused predict+update step moves exactly the algorithmic bytes (record in + record out) through HBM.  The record's
// off-diagonal 8 x 8 tiles are stored in accumulator order: moving one between the record and the DMMA accumulators
// is one conflict-free 16-byte access per lane.
//
// update: the N x N factorisation is a BLOCKED right-looking one in the square-root-free form Pk = U D^-1 U^T
//   (L(:,k) = U(:,k) / sqrt(d_k), see CholStep in slb_predict12.cuh for the scalar version): panels of 4 columns, the
//   trailing matrix lives in FP64 DMMA accumulator tiles (m8n8k4: lane (a = lane & 3, b = lane >> 2) holds entries
//   (8I + b, 8J + 2a) and (8I + b, 8J + 2a + 1) of tile (I, J)), so one panel's rank-4 update is ONE DMMA per tile fed
//   by one shared-memory word per lane and tile row -- the scalar version needed 4 x (rows + cols) words and 4 FMAs
//   per entry.  Per panel: the 16 lanes holding its columns park them in shared memory, every lane redoes the 4 x 4
//   diagonal block's elimination (4 reciprocals, ~20 FMAs -- the same issue slots as one lane doing it), lane t
//   finishes row 8 J0 + t of the panel (6 FMAs; rows above tile row J0 = K >> 3 are zero and are skipped), and the
//   finished rows are both the A and (scaled by -1/d_k) the B fragments.
//   Only the columns that can move h are factored (j < 36 + nk, rounded up to a panel): rows below come out of the same
//   panels (the TRSM is implicit), the trailing block of featuresk_l is never touched.
//   The factor is NOT kept: sigma point j = mu [+] +-L(:,j) needs column j only, so after every 4 panels the 32 sigma
//   points of those 16 columns go through h (one per lane), their contribution to the mean / innovation covariance is
//   accumulated as deviations from Z0 = h(mu) (columns that cannot move h contribute nothing), and
//   covXZ += U(:, 16 cols) W'(16 cols, :) with W'_j = (Z+_j - Z-_j) / (2 sqrt d_j)  (:714-737 without the
//   exp/log round trip, quirk Q10), one DMMA per panel and tile row into covXZ accumulator tiles.
//   K = covXZ S^-1 (:286-288), K S K^T = covXZ K^T; Pk -= covXZ K^T is again one DMMA per tile, on the record in
//   shared memory.
// predict: slb_predict12.cuh's predict12_block on rows 24..35 of the resident record.
#pragma once
#include "slb_predict12.cuh"

namespace slbd {

template <int NK_, int NL_>
struct StepCfg {
    static constexpr int NK = NK_, NL = NL_, NF = NK_ + NL_;
    static constexpr int N = 36 + NK_ + NL_;
    static constexpr int NP = N * (N + 1) / 2;
    static constexpr int PSTR = (NP + 15) / 16 * 16;   // == slb_batch_s::pstride
    static constexpr int QD = 39 + NK_ + NL_;
    static constexpr int QS = (QD + 1) / 2 * 2;        // == slb_batch_s::qstride
    static constexpr int NT = (N + 7) / 8;             // 8 x 8 accumulator tiles per side
    static constexpr int NPAD = 8 * NT;
    static constexpr int JM = 36 + NK_;                // columns j >= JM cannot move h
    static constexpr int NPAN = (JM + 3) / 4;          // panels of 4 columns that are factored
    static constexpr int NCOL = 4 * NPAN;
    static constexpr int JLAST = (NCOL - 1) >> 3;      // last tile column that is ever updated
    static constexpr int NGRP = (NPAN + 3) / 4;        // sigma-point passes (16 columns = 32 points each)
    // A finished panel (NPAD rows x 4 columns) is stored as two planes of column PAIRS, element (i, c) at
    // (c >> 1) * PL + 2 i + (c & 1): row accesses (one double2 per lane and plane) and DMMA fragment loads are then
    // contiguous across the warp.  PL = 8 mod 16 puts the two planes half a bank cycle apart (the 16-lane panel
    // extraction writes both planes in one instruction), and with PS4 = 2 mod 16 the 16 columns of a group fall into 16
    // different bank pairs for the sigma points' column reads: (c & 1) + 8 (c >> 1) + 2 q covers 0..15.
    static constexpr int PL = 2 * NPAD + 8;
    static constexpr int PS4 = 2 * PL + 2;             // stride between the 4 panels of a group
    static constexpr int KP = (NK_ + 3) / 4 * 4;       // padded row length of K / covXZ (DMMA k-dimension)
    static constexpr int NTN = (NK_ + 7) / 8;          // 8-column accumulator tiles of covXZ
    static constexpr int LF = 4 * PS4;                 // finished panel rows U of the current group
    static constexpr int LRAW = 2 * PL;                // the current panel as extracted from the accumulators (same planes)
    static constexpr int KK = 2 * NPAD * KP + NPAD;    // K | covXZ rows | K nu, overlay LF | LRAW once the factorisation is over
    static constexpr int SCR0 = (LF + LRAW > KK ? LF + LRAW : KK);
    // W' of the current group, [c][WS]: the DMMA B fragment W'(K + a, c = b) is then conflict-free (4 c + a covers 0..15)
    static constexpr int WS = 20;
    static constexpr int WGS = WS * NK_;
    static constexpr int UPD_SCR = SCR0 + WGS + NPAD;       // + d_k
    static constexpr int SCR = (UPD_SCR > PRED_SCR ? UPD_SCR : PRED_SCR);
    static constexpr int ZS = (NK_ + 1) / 2 * 2;
    static constexpr int SM = PSTR + QS + SCR + ZS + 2;    // doubles per warp (even); last slot = barrier
    // per-instance noise (the PIN instantiation): the lower triangle of this instance's R, packed, between z and the
    // barrier.  (Its Q entries travel in registers: 6 per lane, see load_q_entries.)
    static constexpr int RP = (NK_ * (NK_ + 1) / 2 + 1) / 2 * 2;
    static constexpr int SMP = SM + RP;
    static_assert(NK_ % 3 == 0 && NK_ >= 3, "the VO model moves 3-D features");
    static_assert(N <= 64, "two rows per lane");
    static_assert(SM % 2 == 0 && PSTR % 2 == 0 && QS % 2 == 0, "16-byte alignment of the bulk copies");
};

// symmetric inverse of the M x M innovation covariance (packed lower in, packed lower out) through its LDL^T
// factorisation, redundantly on every lane; false if a pivot is not positive
template <int M>
SLB_DEV bool sym_inverse(const double *S, double *Si) {
    double L[M * (M + 1) / 2], dd[M], rd[M];   // unit lower L below the diagonal, D and 1 / D
    bool ok = true;
#pragma unroll
    for (int k = 0; k < M; ++k) {
        double d = S[tri(k, k)];
#pragma unroll
        for (int p = 0; p < k; ++p) d = fma(-L[tri(k, p)] * L[tri(k, p)], dd[p], d);
        ok = ok && (d > 0.0);
        dd[k] = d;
        rd[k] = rcp_fast(d);
#pragma unroll
        for (int i = k + 1; i < M; ++i) {
            double s = S[tri(i, k)];
#pragma unroll
            for (int p = 0; p < k; ++p) s = fma(-L[tri(i, p)] * L[tri(k, p)], dd[p], s);
            L[tri(i, k)] = s * rd[k];
        }
    }
    // X = L^-1 (unit lower), Si = X^T D^-1 X
    double X[M * (M + 1) / 2];
#pragma unroll
    for (int j = 0; j < M; ++j) {
        X[tri(j, j)] = 1.0;
#pragma unroll
        for (int i = j + 1; i < M; ++i) {
            double s = 0.0;
#pragma unroll
            for (int p = j; p < i; ++p) s = fma(-L[tri(i, p)], X[tri(p, j)], s);
            X[tri(i, j)] = s;
        }
    }
#pragma unroll
    for (int i = 0; i < M; ++i)
#pragma unroll
        for (int j = 0; j <= i; ++j) {
            double s = 0.0;
#pragma unroll
            for (int k = i; k < M; ++k) s = fma(X[tri(k, i)] * rd[k], X[tri(k, j)], s);
            Si[tri(i, j)] = s;
        }
    return ok;
}

// h of test/UsckfUnitTest.cpp:62-86: delta = statek [-] statek_i as a transform, applied to every 3-D feature
template <int NK>
SLB_DEV void vo_model(const double *pk, const double *qk, const double *pi, const double *qi, const double *f, double *z) {
    double dq[4];
    quat_cmul(qi, qk, dq);
#pragma unroll
    for (int c = 0; c < NK; c += 3) {
        double rz[3];
        rotmat_apply(dq, f + c, rz);
        z[c] = rz[0] + (pk[0] - pi[0]);
        z[c + 1] = rz[1] + (pk[1] - pi[1]);
        z[c + 2] = rz[2] + (pk[2] - pi[2]);
    }
}

template <class C>
struct UpdState {
    double c0[C::NT][C::JLAST + 1], c1[C::NT][C::JLAST + 1];   // accumulator tiles (I >= J)
    double x0[C::NT][C::NTN], x1[C::NT][C::NTN];               // covXZ accumulator tiles (unscaled sum)
    double esum[C::NK], eep[C::NK * (C::NK + 1) / 2];          // sum e, sum e e^T over this lane's sigma points, e = Z - Z0
    double z0[C::NK];
    bool ok;
};

// ---- sigma points of columns 16 G .. 16 G + 15 through h, W' of those columns, covXZ += U W' ---------------------
template <class C, int G>
SLB_DEV void sigma_group(UpdState<C> &s, const double *mus_, const double *Lf, double *Wg, const double *dv, int lane) {
    constexpr int NK = C::NK, PS4 = C::PS4;
    // the mean scalars h needs, as 16-byte broadcast loads (statek pos|quat = mus[0..6], statek_i = mus[26..32])
    double mus[40 + NK];
    {
        const double2 *m2 = reinterpret_cast<const double2 *>(mus_);
#pragma unroll
        for (int e = 0; e < 4; ++e) { const double2 v = m2[e]; mus[2 * e] = v.x; mus[2 * e + 1] = v.y; }
#pragma unroll
        for (int e = 13; e < 17; ++e) { const double2 v = m2[e]; mus[2 * e] = v.x; mus[2 * e + 1] = v.y; }
#pragma unroll
        for (int c = 0; c < NK; ++c) mus[39 + c] = mus_[39 + c];
    }
    constexpr int col0 = 16 * G;
    constexpr int ncols = C::NCOL - col0 < 16 ? C::NCOL - col0 : 16;
    const bool neg = lane & 1, act = (lane >> 1) < ncols;
    const int jl = act ? lane >> 1 : 0;                    // idle lanes (last group) shadow column 0 with a zero scale
    const double rs = rsqrt_fast(dv[col0 + jl]);           // L(:,j) = U(:,j) / sqrt(d_j): the scale rides on the sign
    const double sgn = act ? (neg ? -rs : rs) : 0.0;
    // U(r, j) = col[2 r] for r >= 8 (j >> 3); the rows of tile row j >> 3 above the diagonal hold zeros, the rows above
    // it are not written (finish) and read as zero here.  Rows >= RW are written for every column of the group.
    constexpr int RW = 8 * ((col0 + ncols - 1) >> 3);
    const double *col = Lf + (jl >> 2) * PS4 + ((jl & 3) >> 1) * C::PL + (jl & 1);
    auto Lc = [&](int r) -> double { return sgn * (r >= RW || r >= col0 + jl ? col[2 * r] : 0.0); };
    double xpk[3], xqk[4], xpi[3], xqi[4], xf[NK];
    if (col0 <= 5) {   // column j perturbs rows >= j only: statek is untouched from the second group on
#pragma unroll
        for (int c = 0; c < 3; ++c) xpk[c] = mus[c] + Lc(c);
        const double v[3] = {Lc(3), Lc(4), Lc(5)};
        const double q[4] = {mus[3], mus[4], mus[5], mus[6]};
        double e[4];
        so3_exp(v, 1.0, e);
        quat_mul(q, e, xqk);
    } else {
#pragma unroll
        for (int c = 0; c < 3; ++c) xpk[c] = mus[c];
#pragma unroll
        for (int c = 0; c < 4; ++c) xqk[c] = mus[3 + c];
    }
    if (col0 <= 29) {
#pragma unroll
        for (int c = 0; c < 3; ++c) xpi[c] = mus[26 + c] + Lc(24 + c);
        const double v[3] = {Lc(27), Lc(28), Lc(29)};
        const double q[4] = {mus[29], mus[30], mus[31], mus[32]};
        double e[4];
        so3_exp(v, 1.0, e);
        quat_mul(q, e, xqi);
    } else {
#pragma unroll
        for (int c = 0; c < 3; ++c) xpi[c] = mus[26 + c];
#pragma unroll
        for (int c = 0; c < 4; ++c) xqi[c] = mus[29 + c];
    }
#pragma unroll
    for (int c = 0; c < NK; ++c) xf[c] = mus[39 + c] + Lc(36 + c);
    double z[NK];
    vo_model<NK>(xpk, xqk, xpi, xqi, xf, z);
    double e[NK];
#pragma unroll
    for (int c = 0; c < NK; ++c) {
        e[c] = act ? z[c] - s.z0[c] : 0.0;
        s.esum[c] += e[c];
        const double zp = __shfl_xor_sync(FULL, z[c], 1);
        if (act && !neg) Wg[c * C::WS + jl] = (0.5 * rs) * (z[c] - zp);   // W'_j = (Z+ - Z-) / (2 sqrt d_j)
    }
#pragma unroll
    for (int r = 0; r < NK; ++r)
#pragma unroll
        for (int c = 0; c <= r; ++c) s.eep[tri(r, c)] = fma(e[r], e[c], s.eep[tri(r, c)]);
    __syncwarp();
    // covXZ += U(:, K..K+3) W'(K..K+3, :) for each panel of the group: one DMMA per tile row I >= K >> 3 (the rows above
    // are zero) and covXZ column tile, A = U(8I + b, K + a) as in the rank-4 update, B = W'(K + a, 8T + b), zero beyond nk
    const int a_ = lane & 3, b_ = lane >> 2;
#pragma unroll
    for (int qq = 0; qq < ncols / 4; ++qq) {
        const int J0 = (col0 + 4 * qq) >> 3;
        const double *fp = Lf + qq * PS4 + (a_ >> 1) * C::PL + (a_ & 1) + 2 * b_;
        double w[C::NTN];
#pragma unroll
        for (int T = 0; T < C::NTN; ++T) w[T] = 8 * T + b_ < NK ? Wg[(8 * T + b_) * C::WS + 4 * qq + a_] : 0.0;
#pragma unroll
        for (int I = J0; I < C::NT; ++I) {
            const double f = fp[16 * I];
#pragma unroll
            for (int T = 0; T < C::NTN; ++T) dmma884(s.x0[I][T], s.x1[I][T], f, w[T]);
        }
    }
}

// ---- one panel of 4 columns (compile-time index P), then the group pass after every 4th ---------------------------
template <class C, int P>
struct PanelStep {
    SLB_DEV static void run(UpdState<C> &s, const double *mus, double *Lf, double *Lraw, double *Wg, double *dv, int lane) {
        constexpr int NT = C::NT, JLAST = C::JLAST, PS4 = C::PS4;
        constexpr int K = 4 * P, J0 = K >> 3, H = (K >> 2) & 1, Q = P & 3;
        constexpr int I1 = (K + 4) >> 3;     // first tile row / column with live entries after this panel
        const int a_ = lane & 3, b_ = lane >> 2;
        double *Lq = Lf + Q * PS4;
        constexpr int PL = C::PL;
        // (1) the 16 lanes holding columns K..K+3 park them (rows of tile row J0 and below), a column pair per plane
        if ((a_ >> 1) == H) {
#pragma unroll
            for (int I = J0; I < NT; ++I)
                *reinterpret_cast<double2 *>(Lraw + (a_ & 1) * PL + 2 * (8 * I + b_)) = make_double2(s.c0[I][J0], s.c1[I][J0]);
        }
        __syncwarp();
        // (2) the 4 x 4 diagonal block, eliminated redundantly by every lane
        double m10, m20, m30, m21, m31, m32, r0, r1, r2, r3, d0, d1, d2, d3;
        {
            const double *A = Lraw + 2 * K, *Bp = A + PL;
            const double a00 = A[0];
            const double2 a1 = *reinterpret_cast<const double2 *>(A + 2);
            const double2 a2 = *reinterpret_cast<const double2 *>(A + 4);
            const double a22 = Bp[4];
            const double2 a3 = *reinterpret_cast<const double2 *>(A + 6), a3b = *reinterpret_cast<const double2 *>(Bp + 6);
            d0 = a00;
            r0 = rcp_fast(d0);
            m10 = a1.x * r0; m20 = a2.x * r0; m30 = a3.x * r0;
            d1 = fma(-a1.x, m10, a1.y);
            const double u21 = fma(-a2.x, m10, a2.y), u31 = fma(-a3.x, m10, a3.y);
            r1 = rcp_fast(d1);
            m21 = u21 * r1; m31 = u31 * r1;
            d2 = fma(-u21, m21, fma(-a2.x, m20, a22));
            const double u32 = fma(-u31, m21, fma(-a3.x, m20, a3b.x));
            r2 = rcp_fast(d2);
            m32 = u32 * r2;
            d3 = fma(-u32, m32, fma(-u31, m31, fma(-a3.x, m30, a3b.y)));
            r3 = rcp_fast(d3);
            s.ok = s.ok && (d0 > 0.0) && (d1 > 0.0) && (d2 > 0.0) && (d3 > 0.0);
        }
        if (lane == 0) {
            *reinterpret_cast<double2 *>(dv + K) = make_double2(d0, d1);
            *reinterpret_cast<double2 *>(dv + K + 2) = make_double2(d2, d3);
        }
        // (3) lane t finishes rows 8 J0 + t and 8 J0 + 32 + t of the panel: U(i, K + c), zeros above the diagonal.  The
        //     rows above tile row J0 are zero and are neither written nor read: the fragments below start at I1 >= J0, the
        //     covXZ DMMAs at J0, and the sigma points select zeros there.
        constexpr int R0 = 8 * J0, NLIVE = C::NPAD - R0;
        auto finish = [&](int i) {
            const double2 x01 = *reinterpret_cast<const double2 *>(Lraw + 2 * i);
            const double2 x23 = *reinterpret_cast<const double2 *>(Lraw + PL + 2 * i);
            const double u0 = x01.x;
            const double u1 = fma(-u0, m10, x01.y);
            const double u2 = fma(-u1, m21, fma(-u0, m20, x23.x));
            const double u3 = fma(-u2, m32, fma(-u1, m31, fma(-u0, m30, x23.y)));
            double2 u01, u23;
            u01.x = i >= K ? u0 : 0.0;
            u01.y = i >= K + 1 ? u1 : 0.0;
            u23.x = i >= K + 2 ? u2 : 0.0;
            u23.y = i >= K + 3 ? u3 : 0.0;
            *reinterpret_cast<double2 *>(Lq + 2 * i) = u01;
            *reinterpret_cast<double2 *>(Lq + PL + 2 * i) = u23;
        };
        if (NLIVE >= 32 || lane < NLIVE) finish(R0 + lane);
        if (NLIVE > 32 && lane < NLIVE - 32) finish(R0 + 32 + lane);
        __syncwarp();
        // (4) rank-4 update of the live tiles: A fragment = U(8I + b, K + a), B fragment = -U(8J + b, K + a) / d_{K+a}
        if (I1 <= JLAST) {
            double f[NT];
            const double *fp = Lq + (a_ >> 1) * PL + (a_ & 1) + 2 * b_;
#pragma unroll
            for (int I = I1; I < NT; ++I) f[I] = fp[16 * I];
            const double rlo = (a_ & 1) ? r1 : r0, rhi = (a_ & 1) ? r3 : r2;
            const double nr = -((a_ & 2) ? rhi : rlo);
#pragma unroll
            for (int J = I1; J <= JLAST; ++J) {
                const double g = f[J] * nr;
#pragma unroll
                for (int I = J; I < NT; ++I) dmma884(s.c0[I][J], s.c1[I][J], f[I], g);
            }
        }
        if (Q == 3 || P == C::NPAN - 1) sigma_group<C, (P >> 2)>(s, mus, Lf, Wg, dv, lane);
        PanelStep<C, P + 1>::run(s, mus, Lf, Lraw, Wg, dv, lane);
    }
};
template <class C>
struct PanelStep<C, C::NPAN> {
    SLB_DEV static void run(UpdState<C> &, const double *, double *, double *, double *, double *, int) {}
};

// update of the resident record.  Returns status bits; `dirty` is set when Ps / mus changed, `m2out` (left as it is by
// the early returns) receives the Mahalanobis distance the gate is given.
// PIN: R comes from `Rs`, this instance's packed lower triangle staged in shared memory (cp.async, issued with z).
template <int NK, int NL, bool PIN = false>
SLB_DEV int usckf_update_smem(double *Ps, double *mus, double *scr, const double *zs, const double *Rs,
                              const slb::FilterArgs &a, int lane, bool &dirty, double &m2out) {
    typedef StepCfg<NK, NL> C;
    constexpr int N = C::N, NT = C::NT, NPAD = C::NPAD, JLAST = C::JLAST, KP = C::KP;
    const int a_ = lane & 3, b_ = lane >> 2;
    double *Lf = scr, *Lraw = scr + C::LF, *Ks = scr, *Cs = scr + NPAD * KP, *Wg = scr + C::SCR0, *dv = Wg + C::WGS,
           *dl = Cs + NPAD * KP;
    UpdState<C> s;
    s.ok = true;
    // ---- the lower triangle of Pk from the resident record into the accumulator tiles: an off-diagonal tile is stored
    //      in accumulator order (one 16-byte load per lane), diagonal tiles are filled symmetrically from their packed
    //      triangle, rows / columns beyond N (N % 8 != 0) are an identity block ------------------------------------
    auto elem = [&](int i, int j) -> double {
        if (i >= N || j >= N) return i == j ? 1.0 : 0.0;
        return i >= j ? Ps[prec(N, i, j)] : Ps[prec(N, j, i)];
    };
#pragma unroll
    for (int I = 0; I < NT; ++I)
#pragma unroll
        for (int J = 0; J <= JLAST; ++J)
            if (J < I) {
                double2 v = make_double2(0.0, 0.0);
                if (8 * I + b_ < N) v = *reinterpret_cast<const double2 *>(Ps + prec(N, 8 * I, 8 * J) + 2 * lane);
                s.c0[I][J] = v.x;
                s.c1[I][J] = v.y;
            } else if (J == I) {
                const int i = 8 * I + b_, j = 8 * J + 2 * a_;
                s.c0[I][J] = elem(i, j);
                s.c1[I][J] = elem(i, j + 1);
            }
#pragma unroll
    for (int I = 0; I < NT; ++I)
#pragma unroll
        for (int T = 0; T < C::NTN; ++T) s.x0[I][T] = s.x1[I][T] = 0.0;
#pragma unroll
    for (int c = 0; c < NK; ++c) s.esum[c] = 0.0;
#pragma unroll
    for (int e = 0; e < NK * (NK + 1) / 2; ++e) s.eep[e] = 0.0;
    {   // Z0 = h(mu)
        double pk[3], qk[4], pi[3], qi[4], ft[NK];
#pragma unroll
        for (int c = 0; c < 3; ++c) { pk[c] = mus[c]; pi[c] = mus[26 + c]; }
#pragma unroll
        for (int c = 0; c < 4; ++c) { qk[c] = mus[3 + c]; qi[c] = mus[29 + c]; }
#pragma unroll
        for (int c = 0; c < NK; ++c) ft[c] = mus[39 + c];
        vo_model<NK>(pk, qk, pi, qi, ft, s.z0);
    }
    // ---- factorisation (Eigen::LLT of :577) interleaved with the sigma points (:275-283) -------------------------
    PanelStep<C, 0>::run(s, mus, Lf, Lraw, Wg, dv, lane);
    if (!s.ok) return SLB_ST_CHOL_FAIL;

    // ---- mean / innovation covariance (:280-282) from the deviations e = Z - Z0 -----------------------------------
    constexpr double NS = (double)(2 * N + 1);
    double ebar[NK], S[NK * (NK + 1) / 2];
    if (PIN) {   // the staged R (and z) must have landed, and be visible to the whole warp
        cp_async_wait0();
        __syncwarp();
    }
    auto Rv = [&](int r, int c) { return PIN ? Rs[tri(r, c)] : __ldg(a.R + r * NK + c); };
    if (NK == 3) {   // 3 + 6 sums in one reduce-scatter pass (the d_k slots are dead: every sigma point has been drawn)
        double v[12], o[12];
#pragma unroll
        for (int c = 0; c < 3; ++c) v[c] = s.esum[c];
#pragma unroll
        for (int e = 0; e < 6; ++e) v[3 + e] = s.eep[e];
        v[9] = v[10] = v[11] = 0.0;
        warp_sum12(v, o, dv, lane);
#pragma unroll
        for (int c = 0; c < 3; ++c) ebar[c] = o[c] * (1.0 / NS);
#pragma unroll
        for (int r = 0; r < NK; ++r)
#pragma unroll
            for (int c = 0; c <= r; ++c)
                S[tri(r, c)] = 0.5 * fma(-NS * ebar[r], ebar[c], o[3 + tri(r, c)]) + Rv(r, c);
    } else {
#pragma unroll
        for (int c = 0; c < NK; ++c) ebar[c] = warp_sum(s.esum[c]) * (1.0 / NS);
#pragma unroll
        for (int r = 0; r < NK; ++r)
#pragma unroll
            for (int c = 0; c <= r; ++c)
                S[tri(r, c)] = 0.5 * fma(-NS * ebar[r], ebar[c], warp_sum(s.eep[tri(r, c)])) + Rv(r, c);
    }
    // ---- K = covXZ S^-1 (:286-288), innovation, Mahalanobis gate (:290-294) --------------------------------------
    double Si[NK * (NK + 1) / 2];
    const bool sok = sym_inverse<NK>(S, Si);
    auto SiAt = [&](int r, int c) { return r >= c ? Si[tri(r, c)] : Si[tri(c, r)]; };
    cp_async_wait0();
    __syncwarp();   // z has landed; every lane is done reading Lf / Wg: K | covXZ overlay them
    double nu[NK], sn[NK], m2 = 0.0;
#pragma unroll
    for (int c = 0; c < NK; ++c) nu[c] = zs[c] - (s.z0[c] + ebar[c]);
#pragma unroll
    for (int r = 0; r < NK; ++r) {
        double t = 0.0;
#pragma unroll
        for (int c = 0; c < NK; ++c) t = fma(SiAt(r, c), nu[c], t);
        sn[r] = t;   // S^-1 nu
        m2 = fma(nu[r], t, m2);
    }
    if (!sok) return SLB_ST_CHOL_FAIL;
    m2out = m2;
    if (!chi2_accept(m2, a.gate)) return SLB_ST_GATE_REJECT;
    // covXZ from the accumulator tiles into the rows of Cs, then lane i turns row i into K, -covXZ and K nu
#pragma unroll
    for (int I = 0; I < NT; ++I)
#pragma unroll
        for (int T = 0; T < C::NTN; ++T)
            if (8 * T + 2 * a_ < KP)
                *reinterpret_cast<double2 *>(Cs + (8 * I + b_) * KP + 8 * T + 2 * a_) = make_double2(s.x0[I][T], s.x1[I][T]);
    __syncwarp();
    auto finish_row = [&](int i) {
        double px[NK];
#pragma unroll
        for (int c = 0; c < NK; ++c) px[c] = Cs[i * KP + c];
        double dsum = 0.0;
#pragma unroll
        for (int c = 0; c < KP; ++c) {
            double k = 0.0;
            if (c < NK) {
#pragma unroll
                for (int p = 0; p < NK; ++p) k = fma(px[p], SiAt(p, c), k);
                dsum = fma(px[c], sn[c], dsum);
            }
            Ks[i * KP + c] = k;
            Cs[i * KP + c] = c < NK ? -px[c] : 0.0;   // K S = covXZ: Pk -= covXZ K^T
        }
        dl[i] = dsum;   // (K nu)_i
    };
    finish_row(lane);
    if (lane + 32 < NPAD) finish_row(lane + 32);
    __syncwarp();
    dirty = true;
    // ---- mu = mu [+] K nu (:299-301): lane b < 12 owns block b of the three States, then the feature scalars ------
    bool finite = true;
    if (lane < 12) {
        const int mbw = lane & 3;
        const int mqo = 13 * (lane >> 2) + (mbw == 0 ? 0 : mbw == 1 ? 3 : mbw == 2 ? 7 : 10);
        const double v[3] = {dl[3 * lane], dl[3 * lane + 1], dl[3 * lane + 2]};
        if (mbw == 1) {
            const double q[4] = {mus[mqo], mus[mqo + 1], mus[mqo + 2], mus[mqo + 3]};
            double e[4], o[4];
            so3_exp(v, 1.0, e);
            quat_mul(q, e, o);
#pragma unroll
            for (int c = 0; c < 4; ++c) { mus[mqo + c] = o[c]; finite = finite && isfinite(o[c]); }
        } else {
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                const double o = mus[mqo + c] + v[c];
                mus[mqo + c] = o;
                finite = finite && isfinite(o);
            }
        }
    }
    for (int f = lane; f < NK + NL; f += 32) {
        const double o = mus[39 + f] + dl[36 + f];
        mus[39 + f] = o;
        finite = finite && isfinite(o);
    }
    // ---- Pk -= K S K^T (:296) = Pk - covXZ K^T on the resident record: one DMMA k-step per tile and 4 columns of K
    {
        double fa[NT][KP / 4], fb[NT][KP / 4];
#pragma unroll
        for (int I = 0; I < NT; ++I)
#pragma unroll
            for (int kk = 0; kk < KP / 4; ++kk) {
                fa[I][kk] = Cs[(8 * I + b_) * KP + 4 * kk + a_];
                fb[I][kk] = Ks[(8 * I + b_) * KP + 4 * kk + a_];
            }
#pragma unroll
        for (int I = 0; I < NT; ++I)
#pragma unroll
            for (int J = 0; J <= I; ++J) {
                const int i = 8 * I + b_, j = 8 * J + 2 * a_;
                if (J < I) {   // off-diagonal tile: one 16-byte read-modify-write per lane
                    double2 *pp = reinterpret_cast<double2 *>(Ps + prec(N, 8 * I, 8 * J) + 2 * lane);
                    const bool w = i < N;
                    double2 p = w ? *pp : make_double2(0.0, 0.0);
#pragma unroll
                    for (int kk = 0; kk < KP / 4; ++kk) dmma884(p.x, p.y, fa[I][kk], fb[J][kk]);
                    if (w) *pp = p;
                } else {
                    const bool w0 = i < N && j <= i, w1 = i < N && j + 1 <= i;
                    double p0 = w0 ? Ps[prec(N, i, j)] : 0.0, p1 = w1 ? Ps[prec(N, i, j + 1)] : 0.0;
#pragma unroll
                    for (int kk = 0; kk < KP / 4; ++kk) dmma884(p0, p1, fa[I][kk], fb[J][kk]);
                    if (w0) Ps[prec(N, i, j)] = p0;
                    if (w1) Ps[prec(N, i, j + 1)] = p1;
                }
            }
    }
    return __all_sync(FULL, finite) ? 0 : SLB_ST_NONFINITE;
}

// predict12_block's view of the resident tiled record (rows 24..35 and feature rows 36..)
template <int N>
struct ResidentView {
    static constexpr int ROW0 = 24;
    double *P;
    SLB_DEV int idx(int r, int c) const { return prec(N, 24 + r, c); }
    SLB_DEV double &at(int r, int c) const { return P[idx(r, c)]; }
    SLB_DEV double &feat(int fr, int c) const { return P[prec(N, 36 + fr, 24 + c)]; }
};

// One instance per warp: record in (TMA bulk load), predict and / or update in shared memory, record out (TMA bulk
// store).  PRED && UPD is the fused step (slb_usckf_step, the *_step_host paths); UPD alone is slb_usckf_update.
// PIN: per-instance noise (slb_set_noise_layout), Q at a.Q + inst * a.qs and R at a.R + inst * a.rs (stride 0 = shared).
// Both are fetched with the record: R's lower triangle by cp.async into RP extra doubles of the warp's area, the 6 Q
// entries a lane adds into registers.
// NIS: lane 0 stores the update's m2 to a.nis[inst] (NaN when the update returned before forming it).
template <int PM, int NK, int NL, bool PRED, bool UPD, int WPB, int MINB, bool PIN = false, bool NIS = false>
__global__ void __launch_bounds__(WPB * 32, MINB) usckf_step_kernel(slb::FilterArgs a) {
    typedef StepCfg<NK, NL> C;
    constexpr int SMW = PIN ? C::SMP : C::SM;
    extern __shared__ __align__(128) double smem[];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int inst = blockIdx.x * WPB + w;
    if (inst >= a.B) return;
    double *Ps = smem + (size_t)w * SMW, *mus = Ps + C::PSTR, *scr = mus + C::QS, *zs = scr + C::SCR;
    double *Rs = zs + C::ZS;   // PIN only
    uint64_t *bar = reinterpret_cast<uint64_t *>(zs + C::ZS + (PIN ? C::RP : 0));
    double *Pg = a.P + (size_t)inst * a.pstride;
    double *mug = a.mu + (size_t)inst * a.qstride;
    if (lane == 0) {
        mbar_init(bar, 1);
        mbar_expect_tx(bar, (C::PSTR + C::QS) * 8);
        bulk_g2s(Ps, Pg, C::PSTR * 8, bar);
        bulk_g2s(mus, mug, C::QS * 8, bar);
    }
    // the measurement and the control input are fetched now: with the zero-copy *_step_host they live in mapped host
    // memory and their PCIe latency must not sit in the middle of the step
    if (UPD && lane < NK) {
        cp_async8(zs + lane, a.z + (size_t)inst * NK + lane);
        cp_async_commit();
    }
    if (PIN && UPD) {   // lower triangle of this instance's R, packed (Rs[tri(r, c)])
        const double *Ri = a.R + (size_t)inst * a.rs;
        for (int e = lane; e < NK * (NK + 1) / 2; e += 32) {
            const int r = tri_row(e);
            cp_async8(Rs + e, Ri + r * NK + (e - tri(r, 0)));
        }
        cp_async_commit();
    }
    double qv[PIN && PRED ? 6 : 1];
    if (PIN && PRED) load_q_entries(a.Q + (size_t)inst * a.qs, lane & 3, lane >> 2, qv);
    double u[ProcessModel<PM>::NU];
    if (PRED) {
#pragma unroll
        for (int c = 0; c < ProcessModel<PM>::NU; ++c) u[c] = a.u[(size_t)inst * ProcessModel<PM>::NU + c];
    }
    __syncwarp();
    mbar_wait(bar, 0);
    int st = 0;
    bool dirty = false;
    if (PRED) {
        st = predict12_block<PM, true, PIN>(ResidentView<C::N>{Ps}, mus + 26, u, a.dt, scr, a.Q, qv, NK + NL, mus + 26, lane, dirty);
    }
    double m2 = __longlong_as_double(0x7ff8000000000000ll);   // NaN
    if (UPD) st |= usckf_update_smem<NK, NL, PIN>(Ps, mus, scr, zs, Rs, a, lane, dirty, m2);
    if (NIS && lane == 0) a.nis[inst] = m2;
    cp_async_wait0();   // (an update that bailed out early has not waited for z)
    // ---- record out ----------------------------------------------------------------------------------------------
    if (dirty) {
        fence_proxy_async();
        __syncwarp();
        if (lane == 0) bulk_s2g(Pg, Ps, C::PSTR * 8);
        for (int e = lane; e < C::QD; e += 32) mug[e] = mus[e];
    }
    // optional instance-major copy of the posterior mean (mapped host memory in the zero-copy *_step_host): whatever
    // the step decided (accepted, gated, factorisation failed) the resident record holds the posterior
    if (a.mu_out) {
        __syncwarp();
        for (int e = lane; e < a.out_len; e += 32) a.mu_out[(size_t)inst * a.out_len + e] = mus[a.out_off + e];
    }
    if (st && lane == 0) a.status[inst] |= st;
    if (dirty && lane == 0) bulk_store_wait();
}

}  // namespace slbd
