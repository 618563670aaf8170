// slb_predict12.cuh -- warp-per-instance sigma-point predict of a 12-DOF State block inside a larger
// packed covariance record; shared by Usckf::predict (Usckf.hpp:113-244: block statek_i at rows 24..35,
// cross-covariances propagated) and Msckf::predict (Msckf.hpp:97-189: block statek at rows 0..11, cross
// blocks left stale, quirk Q5).
#pragma once
#include "slb_internal.h"
#include "slb_models.cuh"

namespace slbd {

constexpr unsigned FULL = 0xffffffffu;
SLB_DEV double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(FULL, v, o);
    return v;
}
SLB_DEV double bcast(double v, int src) { return __shfl_sync(FULL, v, src); }

// =====================================================================================================
// 2D-cyclic register layout of a symmetric N x N matrix over one warp and its square-root-free factorisation
// (shared by the USCKF update, N = 36 + nk + nl, and the 12 x 12 predict block)
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

// ---- TMA bulk copy helpers (global -> shared, completion on an mbarrier) ---------------------------
SLB_DEV unsigned saddr(const void *p) { return (unsigned)__cvta_generic_to_shared(p); }
SLB_DEV void mbar_init(uint64_t *bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(saddr(bar)), "r"(count) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
}
SLB_DEV void mbar_expect_tx(uint64_t *bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(saddr(bar)), "r"(bytes) : "memory");
}
SLB_DEV void bulk_g2s(void *dst, const void *src, unsigned bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n" ::"r"(saddr(dst)),
                 "l"(src), "r"(bytes), "r"(saddr(bar))
                 : "memory");
}
SLB_DEV void mbar_wait(uint64_t *bar, unsigned parity) {
    unsigned done = 0;
    while (!done) {
        asm volatile(
            "{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}\n"
            : "=r"(done)
            : "r"(saddr(bar)), "r"(parity)
            : "memory");
    }
}

// D(8x8) += A(8x4) B(4x8) on the FP64 tensor path: lane holds a = A[lane>>2][lane&3], b = B[lane&3][lane>>2] and the
// accumulator pair d0 = D[lane>>2][2*(lane&3)], d1 = D[lane>>2][2*(lane&3)+1].
SLB_DEV void dmma884(double &d0, double &d1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
                 : "+d"(d0), "+d"(d1)
                 : "d"(a), "d"(b));
}

// =====================================================================================================
// predict
// =====================================================================================================
constexpr int PRED_PR = 520;           // USCKF: tile rows 3..4 (rows 24..39), prec(N, 40, 0) - prec(N, 24, 0); MSCKF uses 78 of it
constexpr int PRED_PF = 8 * 12;        // USCKF: 12-wide segments of the feature rows below the span (rows 40..47)
constexpr int PRED_DS = 20;            // row stride of the deviations D and of Fk (= 4 mod 16: conflict-free fragments)
constexpr int PRED_LS = 78 + 16;       // factor, column-major packed (+ pad for the tile overhang)
// doubles per warp (even: 16-B aligned warps for the bulk copy; last slot = mbarrier)
constexpr int PRED_SM = PRED_PR + PRED_PF + PRED_LS + 28 * PRED_DS + 144 + 12 * PRED_DS + 16 + 2;
static_assert(16 * PRED_SM * 8 <= 227 * 1024, "two CTAs of 8 warps per SM");
SLB_DEV void pred_cp_async8(double *smem_dst, const double *gsrc) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;\n" ::"r"(saddr(smem_dst)), "l"(gsrc) : "memory");
}
SLB_DEV void pred_cp_async_wait_all() { asm volatile("cp.async.commit_group;\n cp.async.wait_group 0;\n" ::: "memory"); }

// The 6 entries of a 12 x 12 process noise Q (row-major, lower triangle read) that lane (a_, b_) adds to the predicted
// covariance's DMMA accumulator pairs: rows b_ / 8 + b_, columns 2 a_ (+1) / 8 + 2 a_ (+1); upper-triangle slots are 0.
SLB_DEV void load_q_entries(const double *Qi, int a_, int b_, double *qv) {
    const int rr[6] = {b_, b_, 8 + b_, 8 + b_, 8 + b_, 8 + b_};
    const int cc[6] = {2 * a_, 2 * a_ + 1, 2 * a_, 2 * a_ + 1, 8 + 2 * a_, 9 + 2 * a_};
#pragma unroll
    for (int k = 0; k < 6; ++k) qv[k] = (rr[k] < 12 && cc[k] <= rr[k]) ? __ldg(Qi + rr[k] * 12 + cc[k]) : 0.0;
}

// ROW0: first row of the 12x12 block; MU0: q-vector offset of the block's mean; CROSS: propagate the
// cross-covariances of the block's rows/columns with the rest of the state (USCKF) or not (MSCKF).
//
// The 12 x 12 factorisation is the same square-root-free 2D-cyclic scheme as the USCKF update (CholStep: ~60 cycles
// of serial chain per column instead of the ~280 of a lane-per-row Cholesky built on shuffle broadcasts); every
// rank-k contraction -- the propagated covariance 0.5 D^T D, Fk * P_i,(k|l), P_feat,i * Fk^T -- is 8x8x4 DMMA tiles
// fed straight from shared memory (51 DMMAs replace ~1 100 LDS + DFMA issue slots; rows / columns beyond the block
// only feed accumulator entries that are never stored).
//
// PIN: per-instance Q (slb_set_noise_layout), instance i's 12 x 12 matrix at a.Q + i * a.qs.  Each lane adds at most 6
// entries of Q (put below); it loads exactly those into registers together with the record, so the HBM latency of a
// matrix that no longer sits in L1 overlaps the record's instead of the end of the step.
template <int PM, int WPB, int ROW0, int MU0, bool CROSS, bool PIN = false>
__global__ void __launch_bounds__(WPB * 32, 2) predict12_kernel(slb::FilterArgs a) {
    typedef LayState12 L;
    typedef CycCfg<12> C;
    extern __shared__ __align__(16) double smem[];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int inst = blockIdx.x * WPB + w;
    if (inst >= a.B) return;
    double *Pr = smem + (size_t)w * PRED_SM, *Pf = Pr + PRED_PR, *Ls = Pf + PRED_PF, *D = Ls + PRED_LS, *W = D + 28 * PRED_DS,
           *Fk = W + 144, *rsd = Fk + 12 * PRED_DS;
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
    auto PR = [&](int r, int c) -> double & {   // row ROW0+r, col c
        return Pr[(CROSS ? prec(N, ROW0 + r, c) : tri(ROW0 + r, c)) - T0];
    };
    auto PF = [&](int fr, int c) -> double & {   // feature row fr, col 24 + c
        return fr < NFS ? PR(12 + fr, 24 + c) : Pf[(fr - NFS) * 12 + c];
    };
    const int a_ = lane & 3, b_ = lane >> 2;  // 2D-cyclic tile coordinates == DMMA fragment coordinates (row, k)

    // The block's rows are one contiguous span of the record: one TMA bulk copy (UBLKCP) brings it in, the 12-wide
    // segments of the feature rows below it follow as LDGSTS; the mean and the control input load meanwhile.  The
    // USCKF shapes have N = 39 or N >= 40.
    static_assert((T0 * 8) % 16 == 0 && ((T1 - T0) * 8) % 16 == 0 && PRED_SM % 2 == 0 &&
                      (!CROSS || (((tri(RS, 0) - T0) * 8) % 16 == 0 && ((tri(39, 0) - T0) * 8) % 16 == 0)),
                  "bulk copy needs 16-byte alignment");
    uint64_t *bar = reinterpret_cast<uint64_t *>(rsd + 16);
    if (lane == 0) {
        mbar_init(bar, 1);
        mbar_expect_tx(bar, SPAN * 8);
        bulk_g2s(Pr, Pg + T0, SPAN * 8, bar);
    }
    for (int e = lane; e < nfr * 12; e += 32) {
        const int r = e / 12, c = e - r * 12;
        pred_cp_async8(Pf + e, Pg + prec(N, RS + r, 24 + c));
    }
    double qv[PIN ? 6 : 1];
    if (PIN) load_q_entries(a.Q + (size_t)inst * a.qs, a_, b_, qv);
    double mu[13];
#pragma unroll
    for (int c = 0; c < 13; ++c) mu[c] = mug[MU0 + c];
    ProcessModel<PM> f;
    {
        double u[ProcessModel<PM>::NU];
#pragma unroll
        for (int c = 0; c < ProcessModel<PM>::NU; ++c) u[c] = a.u[(size_t)inst * ProcessModel<PM>::NU + c];
        f.prepare(u, a.dt);
    }
    pred_cp_async_wait_all();
    __syncwarp();
    mbar_wait(bar, 0);

    // ---- Pk_i = U D^-1 U^T (Eigen::LLT of :572-577 up to the per-column scale 1/sqrt(d_k)) ---------------------
    double T[C::RT][C::CT];
#pragma unroll
    for (int r = 0; r < C::RT; ++r)
#pragma unroll
        for (int c = 0; c < C::CT; ++c)
            if (C::exists(r, c)) {
                const int i = a_ + 4 * r, j = b_ + 8 * c;
                T[r][c] = (i < 12 && j <= i) ? PR(i, ROW0 + j) : 0.0;
            }
    bool ok = true;
    {
        const double x0 = __shfl_sync(FULL, T[0][0], 0);
        CholStep<C, 0>::run(T, Ls, a_, b_, ok, x0, -rcp_fast(x0));
    }
    if (!ok) {
        if (lane == 0) a.status[inst] |= SLB_ST_CHOL_FAIL;
        return;
    }
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
        nrm2 = 0.0;
#pragma unroll
        for (int r = 0; r < 12; ++r) {
            md[r] = warp_sum(act ? dd[r] : 0.0) * (1.0 / 25.0);  // not "/ 25.0": zero numerators take div.rn's slow path
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
            for (int r = 0; r < 12; ++r) D[lane * PRED_DS + r] = act ? dY[r] : 0.0;
        }
    }
    __syncwarp();
    // ---- Pk_i = 0.5 D^T D + Q (:178): three lower 8x8 tiles, k = 28 ---------------------------------------------
    {
        double c00[2] = {0.0, 0.0}, c10[2] = {0.0, 0.0}, c11[2] = {0.0, 0.0};
        const double *p0 = D + a_ * PRED_DS + b_, *p1 = p0 + 8;  // A[m][k] = D[k][m]: lane (row b_, k a_)
#pragma unroll
        for (int k0 = 0; k0 < 28; k0 += 4) {
            const double f0 = p0[k0 * PRED_DS], f1 = p1[k0 * PRED_DS];  // columns 12..15 of D: uninitialised, only feed dropped outputs
            dmma884(c00[0], c00[1], f0, f0);
            dmma884(c10[0], c10[1], f1, f0);
            dmma884(c11[0], c11[1], f1, f1);
        }
        // W = 0.5 (dY+ - dY-) is read from D before Pk_i overwrites anything it depends on (D is separate storage)
        if (CROSS) {
            for (int e = lane; e < 144; e += 32) {
                const int jj = e / 12, c = e - jj * 12;
                W[e] = 0.5 * (D[(1 + 2 * jj) * PRED_DS + c] - D[(2 + 2 * jj) * PRED_DS + c]);
            }
        }
        auto put = [&](int r, int c, double v, int k) {
            if (r < 12 && c <= r) PR(r, ROW0 + c) = 0.5 * v + (PIN ? qv[k] : __ldg(a.Q + r * 12 + c));
        };
        const int r = b_, c = 2 * a_;
        put(r, c, c00[0], 0); put(r, c + 1, c00[1], 1);
        put(8 + r, c, c10[0], 2); put(8 + r, c + 1, c10[1], 3);
        put(8 + r, 8 + c, c11[0], 4); put(8 + r, 8 + c + 1, c11[1], 5);
    }
    if (CROSS) {
        __syncwarp();
        // ---- Fk = W^T L^-1  <=>  L^T Fk^T = W: lane c back-substitutes column c (:154); L(p,r) = U(p,r) / sqrt(d_r) --
        if (lane < 12) {
            double x[12];
#pragma unroll
            for (int r = 11; r >= 0; --r) {
                double s = 0.0;
#pragma unroll
                for (int p = r + 1; p < 12; ++p) s = fma(Ls[C::cb(r) - r + p], x[p], s);
                const double rs = rsd[r];
                x[r] = (W[r * 12 + lane] - rs * s) * rs;
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
                    const double bv = PR(k0 + a_, 8 * J + b_);  // B[k][n] = old P(24 + k, n)
                    dmma884(oc[0][J][0], oc[0][J][1], fa0, bv);
                    dmma884(oc[1][J][0], oc[1][J][1], fa1, bv);
                }
            }
        }
        // ---- and with the features (:217-235): feature rows x cols 24..35  <- old * Fk^T: ceil(nf/8) x 2 tiles, k = 12 ----
        double of[4][2][2];
        const int nft = (nf + 7) >> 3;
        {
            const int c0 = min(b_, 11), c1 = min(8 + b_, 11);
#pragma unroll
            for (int I = 0; I < 4; ++I) {
                of[I][0][0] = of[I][0][1] = of[I][1][0] = of[I][1][1] = 0.0;
                if (I < nft) {   // warp-uniform
                    const int fr = min(8 * I + b_, nf - 1);
#pragma unroll
                    for (int k0 = 0; k0 < 12; k0 += 4) {
                        const double av = PF(fr, k0 + a_);
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
                    *reinterpret_cast<double2 *>(Pr + prec(N, ROW0 + 8 * I, 8 * J) - T0 + 2 * lane) =
                        make_double2(oc[I][J][0], oc[I][J][1]);
#pragma unroll
        for (int I = 0; I < 4; ++I)
            if (I < nft) {
#pragma unroll
                for (int J = 0; J < 2; ++J) {
                    const int fr = 8 * I + b_, c = 8 * J + 2 * a_;
                    if (fr < nf && c < 12) { PF(fr, c) = of[I][J][0]; PF(fr, c + 1) = of[I][J][1]; }
                }
            }
        __syncwarp();
    } else {
        __syncwarp();
    }
    // ---- write back --------------------------------------------------------------------------------------
    for (int e = lane; e < SPAN; e += 32) Pg[T0 + e] = Pr[e];
    for (int e = lane; e < nfr * 12; e += 32) {
        const int r = e / 12, c = e - r * 12;
        Pg[prec(N, RS + r, 24 + c)] = Pf[e];
    }
    bool finite = true;
#pragma unroll
    for (int c = 0; c < 13; ++c) {
        finite = finite && isfinite(ref[c]);
        if (lane == c) mug[MU0 + c] = ref[c];
    }
    if (!finite) st |= SLB_ST_NONFINITE;
    if (st && lane == 0) a.status[inst] |= st;
}

}  // namespace slbd
