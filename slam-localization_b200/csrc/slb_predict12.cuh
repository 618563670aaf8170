// slb_predict12.cuh -- warp-per-instance sigma-point predict of a 12-DOF State block inside a larger covariance
// record: Usckf::predict (Usckf.hpp:113-244: block statek_i at rows 24..35 of the tiled record, cross-covariances
// propagated) and Msckf::predict (Msckf.hpp:97-189: block statek at rows 0..11 of the packed record, cross blocks left
// stale, quirk Q5).  One body, predict12_block, works on a shared-memory copy of the rows it touches through a view of
// the record format.  Two fetch strategies feed it: predict12_kernel copies only those rows in and out (slb_usckf_predict,
// slb_msckf_predict), the fused usckf_step_kernel (slb_usckf_step.cuh) runs it on the whole resident record.
#pragma once
#include "slb_internal.h"
#include "slb_models.cuh"
#include "slb_ptx.cuh"

namespace slbd {

// =====================================================================================================
// 2D-cyclic register layout of a symmetric N x N matrix over one warp and its square-root-free factorisation
// (the 12 x 12 predict block)
// =====================================================================================================
template <int N_>
struct CycCfg {
    static constexpr int N = N_;
    static constexpr int RT = (N_ + 3) / 4;      // register tile: rows i = a + 4r, r < RT
    static constexpr int CT = (N_ + 7) / 8;      //                cols j = b + 8c, c < CT
    // first element of column k of the packed column-major factor; L(i,k) = Ls[cb(k) - k + i], i >= k
    SLB_HD static constexpr int cb(int k) { return k * N_ - k * (k - 1) / 2; }
    // tile (r,c) of the 2D-cyclic register layout holds at least one lower-triangular entry
    SLB_HD static constexpr bool exists(int r, int c) { return 4 * r < N_ && 8 * c < N_ && 4 * r + 3 >= 8 * c; }
    // ... and at least one entry (i,j) with j > k (hence i > k): it takes part in the trailing update of step k
    SLB_HD static constexpr bool live(int k, int r, int c) { return exists(r, c) && 8 * c + 7 > k && 4 * r + 3 > k; }
    SLB_HD static constexpr bool row_live(int k, int r) {
        for (int c = 0; c < CT; ++c)
            if (live(k, r, c)) return true;
        return false;
    }
    SLB_HD static constexpr bool col_live(int k, int c) {
        for (int r = 0; r < RT; ++r)
            if (live(k, r, c)) return true;
        return false;
    }
};

// Right-looking factorisation of the N x N covariance held 2D-cyclically in registers: lane (a, b), a = lane & 3,
// b = lane >> 2, owns the entries (a + 4r, b + 8c).  It is computed in the square-root-free form Pk = U D^-1 U^T
// (U = L sqrt(D), unit-free "unscaled" columns: U(i,k) is the Schur-complement entry (i,k) at step k, D = diag U):
// Eigen::LLT's factor is L(:,k) = U(:,k) / sqrt(d_k), a per-column scale that the consumers (sigma points, L W)
// fold into their own per-column coefficients.  What this buys is the length of the serial chain per column: the
// pivot's 1/sqrt no longer sits between the previous trailing update and the publication of the column.  Step K
// (compile-time, fully unrolled by recursion): the 4 lanes holding column K publish it to shared memory as it is
// (column-major packed: exactly the layout the sigma points and L W need afterwards), every lane rank-1-updates
// its live tiles with U(i,K) and -U(j,K)/d_K read back from that column.  -1/d_K arrives from the previous step
// (look-ahead: d_{K+1} = T(K+1,K+1) - U(K+1,K)^2/d_K is formed redundantly by all lanes from one broadcast of
// the old diagonal entry, with the same operations as the owner's tile update so both agree bitwise), so the
// reciprocal's latency overlaps the trailing update.  Entries of finished columns / of the upper triangle are
// never read again, so the update needs no predicate at all: whole tiles are pruned at compile time and the rest
// is plain DFMA.
template <class C, int K>
struct CholStep {
    template <class Tile>
    SLB_DEV static void run(Tile &T, double *Ls, int a_, int b_, bool &ok, double x, double nrcp) {
        constexpr int N = C::N, RT = C::RT, CT = C::CT;
        constexpr int rk = K >> 2, bk = K & 7, ck = K >> 3;
        constexpr int K1 = K + 1 < N ? K + 1 : K;
        constexpr int owner1 = (K1 & 3) + 4 * (K1 & 7);
        constexpr int base = C::cb(K) - K;
        ok = ok && (x > 0.0);
        const double xn_old = __shfl_sync(FULL, T[K1 >> 2][K1 >> 3], owner1);
#pragma unroll
        for (int r = rk; r < RT; ++r) {
            const int i = a_ + 4 * r;
            if (b_ == bk && i >= K && i < N) Ls[base + i] = T[r][ck];
        }
        __syncwarp();
        double li[RT], lj[CT];
#pragma unroll
        for (int r = 0; r < RT; ++r)
            if (C::row_live(K, r)) li[r] = Ls[base + a_ + 4 * r];
#pragma unroll
        for (int c = 0; c < CT; ++c)
            if (C::col_live(K, c)) lj[c] = Ls[base + b_ + 8 * c] * nrcp;
        double xn = x, nrcpn = nrcp;
        if (K + 1 < N) {
            const double u1 = Ls[base + K + 1];
            xn = fma(u1, u1 * nrcp, xn_old);
            nrcpn = -rcp_fast(xn);
        }
#pragma unroll
        for (int r = 0; r < RT; ++r)
#pragma unroll
            for (int c = 0; c < CT; ++c)
                if (C::live(K, r, c)) T[r][c] = fma(li[r], lj[c], T[r][c]);
        CholStep<C, K + 1>::run(T, Ls, a_, b_, ok, xn, nrcpn);
    }
};
template <class C>
struct CholStep<C, C::N> {
    template <class Tile>
    SLB_DEV static void run(Tile &, double *, int, int, bool &, double, double) {}
};

// =====================================================================================================
// predict
// =====================================================================================================
// Scratch of one predict, per warp: Ls | D | W | Fk | rsd | slots.
constexpr int PRED_DS = 20;            // row stride of the deviations D and of Fk (= 4 mod 16: conflict-free fragments)
constexpr int PRED_LS = 78 + 16;       // factor, column-major packed (+ pad for the tile overhang)
constexpr int PRED_D = 28 * PRED_DS;   // deviations: 25 sigma points + 3 zero rows of DMMA k-padding
constexpr int PRED_W = 144;            // W = 0.5 (dY+ - dY-), 12 x 12
constexpr int PRED_FK = 12 * PRED_DS;  // Fk
constexpr int PRED_RSD = 16;           // 1 / L_kk
constexpr int PRED_SLOTS = 16;         // warp_sum12's partial sums
constexpr int PRED_SCR = PRED_LS + PRED_D + PRED_W + PRED_FK + PRED_RSD + PRED_SLOTS;
// predict12_kernel's partial record, per warp: the span | the feature rows below it | scratch | mean, input | barrier
constexpr int PRED_PR = 520;           // USCKF: tile rows 3..4 (rows 24..39), prec(N, 40, 0) - prec(N, 24, 0); MSCKF uses 78 of it
constexpr int PRED_PF = 8 * 12;        // USCKF: 12-wide segments of the feature rows below the span (rows 40..47)
constexpr int PRED_MU = 26;            // the mean (13) and the control input (up to 13), staged by cp.async
constexpr int PRED_SM = PRED_PR + PRED_PF + PRED_SCR + PRED_MU + 2;   // doubles per warp (even: 16-B aligned warps for the bulk copy)
static_assert(16 * PRED_SM * 8 <= 227 * 1024, "two CTAs of 8 warps per SM");

// The 6 entries of a 12 x 12 process noise Q (row-major, lower triangle read) that lane (a_, b_) adds to the predicted
// covariance's DMMA accumulator pairs: rows b_ / 8 + b_, columns 2 a_ (+1) / 8 + 2 a_ (+1); upper-triangle slots are 0.
SLB_DEV void load_q_entries(const double *Qi, int a_, int b_, double *qv) {
    const int rr[6] = {b_, b_, 8 + b_, 8 + b_, 8 + b_, 8 + b_};
    const int cc[6] = {2 * a_, 2 * a_ + 1, 2 * a_, 2 * a_ + 1, 8 + 2 * a_, 9 + 2 * a_};
#pragma unroll
    for (int k = 0; k < 6; ++k) qv[k] = (rr[k] < 12 && cc[k] <= rr[k]) ? __ldg(Qi + rr[k] * 12 + cc[k]) : 0.0;
}

// Sums of 12 values over the 32 lanes, result on every lane.  A butterfly per value costs 5 shuffles each (120 SHFL.32 for
// 12 doubles, and shuffles travel through the same data pipe as shared memory, the fused step's limiter); here the lanes
// halve the VALUE set while they halve the lane set (8 + 4 + 2 + 1 + 1 exchanges), the 16 partial owners park their sums
// in shared memory and everybody reads them back with broadcast loads: 32 SHFL.32 + 1 STS + 6 LDS.128.  The additions
// pair the same partners in the same order as warp_sum's butterfly, so each sum is bitwise warp_sum's.
SLB_DEV void warp_sum12(const double *v, double *out, double *slots, int lane) {
    double a[8], b[4], c[2], d1;
    const bool h16 = lane & 16, h8 = lane & 8, h4 = lane & 4, h2 = lane & 2;
#pragma unroll
    for (int i = 0; i < 8; ++i) {   // values 12..15 are zero padding
        const double lo = v[i], hi = i < 4 ? v[8 + i] : 0.0;
        const double r = __shfl_xor_sync(FULL, h16 ? lo : hi, 16);
        a[i] = (h16 ? hi : lo) + r;                     // lanes < 16 own values 0..7, lanes >= 16 own 8..15
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const double r = __shfl_xor_sync(FULL, h8 ? a[i] : a[4 + i], 8);
        b[i] = (h8 ? a[4 + i] : a[i]) + r;
    }
#pragma unroll
    for (int i = 0; i < 2; ++i) {
        const double r = __shfl_xor_sync(FULL, h4 ? b[i] : b[2 + i], 4);
        c[i] = (h4 ? b[2 + i] : b[i]) + r;
    }
    {
        const double r = __shfl_xor_sync(FULL, h2 ? c[0] : c[1], 2);
        d1 = (h2 ? c[1] : c[0]) + r;
    }
    d1 += __shfl_xor_sync(FULL, d1, 1);
    // value index owned by this lane: bit 3 = h16, bit 2 = h8, bit 1 = h4, bit 0 = h2
    const int idx = (h16 ? 8 : 0) + (h8 ? 4 : 0) + (h4 ? 2 : 0) + (h2 ? 1 : 0);
    __syncwarp();
    if (!(lane & 1)) slots[idx] = d1;
    __syncwarp();
#pragma unroll
    for (int i = 0; i < 6; ++i) {
        const double2 t = *reinterpret_cast<const double2 *>(slots + 2 * i);
        out[2 * i] = t.x;
        out[2 * i + 1] = t.y;
    }
}

// One predict of a 12 x 12 State block, one warp.  The View hides the record's format: v.at(r, c) = v.P[v.idx(r, c)] is
// entry (ROW0 + r, c) of the covariance, r < 12, c < ROW0 + 12 (View::ROW0: the block's first row and column),
// v.feat(fr, c) entry (ROW0 + 12 + fr, ROW0 + c) of feature row fr (CROSS only).  Off-diagonal 8 x 8 tiles of the rows
// ROW0.. must be row-major (the tiled record, prec): a cross-covariance tile is stored as one 16-byte access per lane.
// CROSS: propagate the cross-covariances of the block's rows / columns with the rest of the state (USCKF, nf feature
// rows) or not (MSCKF).  mu_src: the block's 13 mean scalars in shared memory (mu_dst may be the same address);
// u, dt: the process model's input.  The mean is read and the model prepared here rather than by the callers:
// that keeps the fused step's instruction schedule.  PIN: Q comes from qv, the 6 entries this lane adds
// (load_q_entries), instead of the shared matrix at Qg.
//
// The 12 x 12 factorisation is the square-root-free 2D-cyclic CholStep (~60 cycles of serial chain per column instead of
// the ~280 of a lane-per-row Cholesky built on shuffle broadcasts); every rank-k contraction -- the propagated
// covariance 0.5 D^T D, Fk * P_i,(k|l), P_feat,i * Fk^T -- is 8x8x4 DMMA tiles fed straight from shared memory (51 DMMAs
// replace ~1 100 LDS + DFMA issue slots; rows / columns beyond the block only feed accumulator entries that are never
// stored).
//
// Returns status bits.  On SLB_ST_CHOL_FAIL it returns before writing anything; otherwise `dirty` is set, the block, its
// cross-covariances and the 13 mean scalars at mu_dst hold the prediction, and the warp has synchronised.
template <int PM, bool CROSS, bool PIN, class View>
SLB_DEV int predict12_block(View v, const double *mu_src, const double *u, double dt, double *scr, const double *Qg,
                            const double *qv, int nf, double *mu_dst, int lane, bool &dirty) {
    typedef LayState12 L;
    typedef CycCfg<12> C;
    constexpr int ROW0 = View::ROW0;
    double *Ls = scr, *D = Ls + PRED_LS, *W = D + PRED_D, *Fk = W + PRED_W, *rsd = Fk + PRED_FK, *slots = rsd + PRED_RSD;
    const int a_ = lane & 3, b_ = lane >> 2;  // 2D-cyclic tile coordinates == DMMA fragment coordinates (row, k)
    double mu[13];
#pragma unroll
    for (int c = 0; c < 13; ++c) mu[c] = mu_src[c];
    ProcessModel<PM> f;
    f.prepare(u, dt);
    // ---- Pk_i = U D^-1 U^T (Eigen::LLT of :572-577 up to the per-column scale 1/sqrt(d_k)) ---------------------
    double T[C::RT][C::CT];
#pragma unroll
    for (int r = 0; r < C::RT; ++r)
#pragma unroll
        for (int c = 0; c < C::CT; ++c)
            if (C::exists(r, c)) {
                const int i = a_ + 4 * r, j = b_ + 8 * c;
                T[r][c] = (i < 12 && j <= i) ? v.at(i, ROW0 + j) : 0.0;
            }
    bool ok = true;
    {
        const double x0 = __shfl_sync(FULL, T[0][0], 0);
        CholStep<C, 0>::run(T, Ls, a_, b_, ok, x0, -rcp_fast(x0));
    }
    if (!ok) return SLB_ST_CHOL_FAIL;
    __syncwarp();
    if (lane < 12) {
        double sq_, rs_;
        sqrt_rsqrt(Ls[C::cb(lane)], sq_, rs_);
        rsd[lane] = rs_;  // 1 / L_kk
    }
    __syncwarp();
    // ---- sigma point `lane` (Usckf.hpp:572-598), process model (:141) ---------------------------------
    const bool act = lane < 25;
    const int j = lane >= 1 ? (lane - 1) >> 1 : 0, jc = j < 12 ? j : 11;
    double Y[13];
    {
        const double sgn = (lane & 1) ? rsd[jc] : -rsd[jc];
        const int cj = C::cb(jc) - jc;
        double d[12], X[13];
#pragma unroll
        for (int r = 0; r < 12; ++r) d[r] = (act && lane >= 1 && r >= jc) ? sgn * Ls[cj + r] : 0.0;
        boxplus<L>(mu, d, 1.0, X);
        f.apply(X, Y);
    }
    // ---- manifold mean (:601-627) --------------------------------------------------------------------
    double ref[13];
#pragma unroll
    for (int c = 0; c < 13; ++c) ref[c] = bcast(Y[c], 0);
    int it = 0;
    double nrm2;
    do {
        double dd[12], md[12], nr[13];
        boxminus<L>(Y, ref, dd);
#pragma unroll
        for (int r = 0; r < 12; ++r) dd[r] = act ? dd[r] : 0.0;
        warp_sum12(dd, md, slots, lane);
        nrm2 = 0.0;
#pragma unroll
        for (int r = 0; r < 12; ++r) {
            md[r] *= (1.0 / 25.0);  // not "/ 25.0": zero numerators take div.rn's slow path
            nrm2 += md[r] * md[r];
        }
        boxplus<L>(ref, md, 1.0, nr);
#pragma unroll
        for (int c = 0; c < 13; ++c) ref[c] = nr[c];
    } while (sqrt(nrm2) > 1e-6 && ++it < 10000);
    int st = (it >= 10000) ? SLB_ST_MEAN_NOCONV : 0;
    {   // deviations, one row per sigma point; rows 25..27 are the zero padding of the DMMA k-dimension
        double dY[12];
        boxminus<L>(Y, ref, dY);
        if (lane < 28) {
#pragma unroll
            for (int r = 0; r < 12; r += 2)   // (row stride 160 B: 16-byte stores, 2-way instead of 8-way bank conflicts)
                *reinterpret_cast<double2 *>(D + lane * PRED_DS + r) = act ? make_double2(dY[r], dY[r + 1]) : make_double2(0.0, 0.0);
        }
    }
    __syncwarp();
    dirty = true;
    // ---- Pk_i = 0.5 D^T D + Q (:178): three lower 8x8 tiles, k = 28 ---------------------------------------------
    {
        double c00[2] = {0.0, 0.0}, c10[2] = {0.0, 0.0}, c11[2] = {0.0, 0.0};
        const double *p0 = D + a_ * PRED_DS + b_, *p1 = p0 + 8;  // A[m][k] = D[k][m]: lane (row b_, k a_)
#pragma unroll
        for (int k0 = 0; k0 < 28; k0 += 4) {
            const double f0 = p0[k0 * PRED_DS], f1 = p1[k0 * PRED_DS];  // columns 12..15 of D only feed dropped outputs
            dmma884(c00[0], c00[1], f0, f0);
            dmma884(c10[0], c10[1], f1, f0);
            dmma884(c11[0], c11[1], f1, f1);
        }
        if (CROSS) {
            for (int e = lane; e < 144; e += 32) {
                const int jj = e / 12, c = e - jj * 12;
                W[e] = 0.5 * (D[(1 + 2 * jj) * PRED_DS + c] - D[(2 + 2 * jj) * PRED_DS + c]);
            }
            __syncwarp();   // the old block (rows ROW0.., cols ROW0..) was consumed by the factorisation: overwrite it
        }
        auto put = [&](int r, int c, double x, int k) {
            if (r < 12 && c <= r) v.at(r, ROW0 + c) = 0.5 * x + (PIN ? qv[k] : __ldg(Qg + r * 12 + c));
        };
        const int r = b_, c = 2 * a_;
        put(r, c, c00[0], 0); put(r, c + 1, c00[1], 1);
        put(8 + r, c, c10[0], 2); put(8 + r, c + 1, c10[1], 3);
        put(8 + r, 8 + c, c11[0], 4); put(8 + r, 8 + c + 1, c11[1], 5);
    }
    if constexpr (CROSS) {
        // ---- Fk = W^T L^-1  <=>  L^T Fk^T = W: lane c back-substitutes column c (:154); L(p,r) = U(p,r) / sqrt(d_r) --
        if (lane < 12) {
            double x[12];
#pragma unroll
            for (int r = 11; r >= 0; --r) {
                double sacc = 0.0;
#pragma unroll
                for (int p = r + 1; p < 12; ++p) sacc = fma(Ls[C::cb(r) - r + p], x[p], sacc);
                const double rs = rsd[r];
                x[r] = (W[r * 12 + lane] - rs * sacc) * rs;
            }
#pragma unroll
            for (int r = 0; r < 12; ++r) Fk[lane * PRED_DS + r] = x[r];
        }
        __syncwarp();
        // ---- cross-covariances with the clones (:191-208): rows 24..35 x cols 0..23  <- Fk * old: 2 x 3 tiles, k = 12 ----
        double oc[2][3][2];
        {
            const int r0 = min(b_, 11), r1 = min(8 + b_, 11);
#pragma unroll
            for (int I = 0; I < 2; ++I)
#pragma unroll
                for (int J = 0; J < 3; ++J) oc[I][J][0] = oc[I][J][1] = 0.0;
#pragma unroll
            for (int k0 = 0; k0 < 12; k0 += 4) {
                const double fa0 = Fk[r0 * PRED_DS + k0 + a_], fa1 = Fk[r1 * PRED_DS + k0 + a_];
#pragma unroll
                for (int J = 0; J < 3; ++J) {
                    const double bv = v.at(k0 + a_, 8 * J + b_);  // B[k][n] = old P(24 + k, n)
                    dmma884(oc[0][J][0], oc[0][J][1], fa0, bv);
                    dmma884(oc[1][J][0], oc[1][J][1], fa1, bv);
                }
            }
        }
        // ---- and with the features (:217-235): feature rows x cols 24..35  <- old * Fk^T: ceil(nf/8) x 2 tiles, k = 12 ----
        // (nf <= 28: N <= 64.  A caller with a compile-time nf gets the tile loops folded to its NFT tiles.)
        const int nft = (nf + 7) >> 3;
        double of[4][2][2];
        {
            const int c0 = min(b_, 11), c1 = min(8 + b_, 11);
#pragma unroll
            for (int I = 0; I < 4; ++I) {
                if (I < nft) {   // warp-uniform
                    of[I][0][0] = of[I][0][1] = of[I][1][0] = of[I][1][1] = 0.0;
                    const int fr = min(8 * I + b_, nf - 1);
#pragma unroll
                    for (int k0 = 0; k0 < 12; k0 += 4) {
                        const double av = v.feat(fr, k0 + a_);
                        dmma884(of[I][0][0], of[I][0][1], av, Fk[c0 * PRED_DS + k0 + a_]);  // B[k][n] = Fk[n][k]
                        dmma884(of[I][1][0], of[I][1][1], av, Fk[c1 * PRED_DS + k0 + a_]);
                    }
                }
            }
        }
        __syncwarp();
        // rows 24..35 x cols 0..23 are off-diagonal tiles of tile rows 3 and 4: one 16-byte store per lane and tile
#pragma unroll
        for (int I = 0; I < 2; ++I)
#pragma unroll
            for (int J = 0; J < 3; ++J)
                if (8 * I + b_ < 12)
                    *reinterpret_cast<double2 *>(v.P + v.idx(8 * I, 8 * J) + 2 * lane) = make_double2(oc[I][J][0], oc[I][J][1]);
#pragma unroll
        for (int I = 0; I < 4; ++I) {
            if (I < nft) {
#pragma unroll
                for (int J = 0; J < 2; ++J) {
                    const int fr = 8 * I + b_, c = 8 * J + 2 * a_;
                    if (fr < nf && c < 12) { v.feat(fr, c) = of[I][J][0]; v.feat(fr, c + 1) = of[I][J][1]; }
                }
            }
        }
    }
    bool finite = true;
#pragma unroll
    for (int c = 0; c < 13; ++c) {
        finite = finite && isfinite(ref[c]);
        if (lane == c) mu_dst[c] = ref[c];
    }
    if (!finite) st |= SLB_ST_NONFINITE;
    __syncwarp();
    return st;
}

// predict12_kernel's views of the block's rows, copied to shared memory at P (record index - first index of row ROW0):
// tile rows 3..4 of a tiled USCKF record (rows 24..39), with the feature rows below them at Pf, 12 wide (columns 24..35)
struct SpanView {
    static constexpr int ROW0 = 24;
    double *P, *Pf;
    int N;
    SLB_DEV int idx(int r, int c) const { return prec(N, 24 + r, c) - tri(24, 0); }
    SLB_DEV double &at(int r, int c) const { return P[idx(r, c)]; }
    SLB_DEV double &feat(int fr, int c) const { return fr < 4 ? at(12 + fr, 24 + c) : Pf[(fr - 4) * 12 + c]; }
};
// rows ROW0..ROW0 + 11 of a packed MSCKF record (tri)
template <int ROW0_>
struct PackedView {
    static constexpr int ROW0 = ROW0_;
    double *P;
    SLB_DEV int idx(int r, int c) const { return tri(ROW0 + r, c) - tri(ROW0, 0); }
    SLB_DEV double &at(int r, int c) const { return P[idx(r, c)]; }
};

// Standalone predict (slb_usckf_predict: CROSS, ROW0 = 24, MU0 = 26; slb_msckf_predict: ROW0 = MU0 = 0), one instance
// per warp.  It fetches only the rows the predict touches -- USCKF tile rows 3..4 and the 12-wide segments of the feature
// rows below, MSCKF rows 0..11 -- runs predict12_block on them and writes them back.
// ROW0: first row of the 12x12 block; MU0: q-vector offset of the block's mean.
// PIN: per-instance Q (slb_set_noise_layout), instance i's 12 x 12 matrix at a.Q + i * a.qs.  Each lane adds at most 6
// entries of Q; it loads exactly those into registers together with the record, so the HBM latency of a matrix that no
// longer sits in L1 overlaps the record's instead of the end of the step.
template <int PM, int WPB, int ROW0, int MU0, bool CROSS, bool PIN = false>
__global__ void __launch_bounds__(WPB * 32, 2) predict12_kernel(slb::FilterArgs a) {
    extern __shared__ __align__(16) double smem[];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int inst = blockIdx.x * WPB + w;
    if (inst >= a.B) return;
    double *Pr = smem + (size_t)w * PRED_SM, *Pf = Pr + PRED_PR, *scr = Pf + PRED_PF;
    double *mus = scr + PRED_SCR, *us = mus + 13;
    uint64_t *bar = reinterpret_cast<uint64_t *>(mus + PRED_MU);
    // USCKF (CROSS) records are tiled (prec): the block's rows 24..35 lie in tile rows 3 and 4, which the span covers
    // whole (rows 24..min(N, 40) - 1, feature rows 36..39 included); MSCKF records are packed (tri): rows ROW0..ROW0+11.
    static_assert(!CROSS || ROW0 == 24, "the tiled span is tile rows 3..4");
    const int nf = CROSS ? a.nk + a.nl : 0, N = CROSS ? 36 + nf : ROW0 + 12;
    constexpr int T0 = ROW0 * (ROW0 + 1) / 2, T1 = (ROW0 + 12) * (ROW0 + 13) / 2;
    constexpr int RS = CROSS ? 40 : ROW0 + 12;         // first record row after the span
    constexpr int NFS = RS - 36;                        // CROSS: feature rows inside the span
    const int SPAN = CROSS ? tri(min(N, RS), 0) - T0 : T1 - T0;
    const int nfr = CROSS && nf > NFS ? nf - NFS : 0;   // feature rows below the span
    static_assert(tri(RS, 0) - T0 <= PRED_PR && (!CROSS || 12 * (48 - RS) <= PRED_PF), "row span");
    double *Pg = a.P + (size_t)inst * a.pstride;
    double *mug = a.mu + (size_t)inst * a.qstride;
    const int a_ = lane & 3, b_ = lane >> 2;

    // The block's rows are one contiguous span of the record: one TMA bulk copy (UBLKCP) brings it in, the 12-wide
    // segments of the feature rows below it, the mean and the control input follow as LDGSTS (staged in shared memory,
    // they hold no registers across the wait).  The USCKF shapes have N = 39 or N >= 40.
    static_assert((T0 * 8) % 16 == 0 && ((T1 - T0) * 8) % 16 == 0 && PRED_SM % 2 == 0 &&
                      (!CROSS || (((tri(RS, 0) - T0) * 8) % 16 == 0 && ((tri(39, 0) - T0) * 8) % 16 == 0)),
                  "bulk copy needs 16-byte alignment");
    if (lane == 0) {
        mbar_init(bar, 1);
        mbar_expect_tx(bar, SPAN * 8);
        bulk_g2s(Pr, Pg + T0, SPAN * 8, bar);
    }
    for (int e = lane; e < nfr * 12; e += 32) {
        const int r = e / 12, c = e - r * 12;
        cp_async8(Pf + e, Pg + prec(N, RS + r, 24 + c));
    }
    double qv[PIN ? 6 : 1];
    if (PIN) load_q_entries(a.Q + (size_t)inst * a.qs, a_, b_, qv);
    static_assert(ProcessModel<PM>::NU <= PRED_MU - 13, "control input slots");
    if (lane < 13) cp_async8(mus + lane, mug + MU0 + lane);
    if (lane < ProcessModel<PM>::NU) cp_async8(us + lane, a.u + (size_t)inst * ProcessModel<PM>::NU + lane);
    cp_async_wait_all();
    __syncwarp();
    mbar_wait(bar, 0);

    int st;
    bool dirty = false;
    if constexpr (CROSS) st = predict12_block<PM, true, PIN>(SpanView{Pr, Pf, N}, mus, us, a.dt, scr, a.Q, qv, nf, mug + MU0, lane, dirty);
    else st = predict12_block<PM, false, PIN>(PackedView<ROW0>{Pr}, mus, us, a.dt, scr, a.Q, qv, nf, mug + MU0, lane, dirty);
    if (dirty) {
        for (int e = lane; e < SPAN; e += 32) Pg[T0 + e] = Pr[e];
        for (int e = lane; e < nfr * 12; e += 32) {
            const int r = e / 12, c = e - r * 12;
            Pg[prec(N, RS + r, 24 + c)] = Pf[e];
        }
    }
    if (st && lane == 0) a.status[inst] |= st;
}

}  // namespace slbd
