// slb_ukf.cu -- ukfom::ukf<state> predict / update / fused step, G lanes per filter instance.
//
// Replaces (per instance) ukfom::ukf::predict / update / apply_delta as exercised at
// test/UKFoMUnitTest.cpp:104-117, whose skeleton is the single-state path of Msckf.hpp
// (:435-496 sigma points + manifold mean, :554-570 covariance, :612-633 cross-covariance,
// :668-675 applyDelta).
//
// Mapping (see DESIGN.md "UKF kernel"):
//   * G = 4 consecutive lanes own one instance, a warp owns 32/G = 8 instances and never talks to
//     another warp (only __syncwarp / shuffles): the on-chip footprint of an instance (its 2n+1
//     propagated sigma points, P, L) bounds how many instances an SM can hold (~100), so the lanes
//     per instance -- not the instances -- supply the warps that hide FP64 latency;
//   * state is SoA in HBM: mu[c][stride], P[e][stride] with P packed lower-triangular; a warp reads
//     8 consecutive instances of G fields per load (64-byte segments);
//   * sigma point s of an instance is handled by lane s % G: drawn from the Cholesky column, pushed
//     through the model and parked in shared memory as Y[c][s] (component-major: the G lanes of a
//     group touch consecutive doubles, groups sit 4 banks apart, so the traffic is conflict-free);
//   * manifold mean: per-lane partial sums of X_s [-] ref, xor-shuffle inside the group, every lane
//     applies the same [+]; covariance: per-lane 0.5 sum d d^T partials in registers, reduced through
//     shared scratch in fixed lane order (bitwise reproducible whatever the batch size);
//   * the 9x9 Cholesky runs redundantly on the G lanes in registers (same issue slots as one lane
//     doing it, no exchange), pivots through MUFU.RSQ64H + Newton;
//   * predict+update fused in one launch moves each instance through HBM exactly once.
#include "slb_internal.h"
#include "slb_models.cuh"
#include "slb_ptx.cuh"

namespace slbd {

template <int G>
SLB_DEV double gsum(double v) {
#pragma unroll
    for (int o = G / 2; o > 0; o >>= 1) v += __shfl_xor_sync(FULL, v, o);
    return v;
}

// In-register packed Cholesky (lower, row-major packed), pivots through sqrt_rsqrt.  Every loop has the
// constant trip count N with compile-time predicates: nvcc then unrolls all three levels and the
// matrix stays in registers (data-dependent bounds left a rolled loop over a local-memory array).
template <int N>
SLB_DEV bool chol_packed_fast(double *A) {
    bool ok = true;
#pragma unroll
    for (int k = 0; k < N; ++k) {
        double x = A[tri(k, k)];
#pragma unroll
        for (int p = 0; p < N; ++p)
            if (p < k) x = fma(-A[tri(k, p)], A[tri(k, p)], x);
        ok = ok && (x > 0.0);
        double sx, inv;
        sqrt_rsqrt(x, sx, inv);
        A[tri(k, k)] = sx;
#pragma unroll
        for (int i = 0; i < N; ++i) {
            if (i > k) {
                double s = A[tri(i, k)];
#pragma unroll
                for (int p = 0; p < N; ++p)
                    if (p < k) s = fma(-A[tri(i, p)], A[tri(k, p)], s);
                A[tri(i, k)] = s * inv;
            }
        }
    }
    return ok;
}

// Shared-memory record of one instance (doubles).  IS = G (mod 16) keeps the G-lane groups of a
// half-warp on disjoint banks for the Y[c][s] accesses.
template <class L, int M, int G>
struct Rec {
    static constexpr int N = L::N, QD = L::QD, NP = L::NP, NS = 2 * L::N + 1;
    static constexpr int UPD_SCR = NS * M + 3 * N * M + N;  // Z | DZ | K | KS | delta
    static constexpr int A0 = NS * QD > UPD_SCR ? NS * QD : UPD_SCR;
    static constexpr int SIGSZ = A0 > G * NP ? A0 : G * NP;  // also the covariance reduction scratch
    static constexpr int SIG = 0, LF = SIGSZ, PS = LF + NP, MU = PS + NP, FLAG = MU + QD;
    static constexpr int UZ = SIG;        // control input u (<= 6) and measurement z (M) are staged in the (not yet live)
                                          // sigma-point area and picked up into registers before it is first written
    static constexpr int RAW = FLAG + 1;
    static constexpr int IS = RAW + ((G - RAW % 16) % 16 + 16) % 16;
    // update scratch inside SIG
    static constexpr int ZO = 0, DZO = NS * M, KO = DZO + N * M, KSO = KO + N * M, DLO = KSO + N * M;
};

// doubles of shared memory per warp: 32/G records, the packed Q, and (16-byte aligned) a barrier slot (mbar_init)
template <class L, int M, int G>
struct UkfWarp {
    static constexpr int DOUBLES = ((32 / G) * Rec<L, M, G>::IS + L::NP + 1) / 2 * 2 + 2;
};

// Cholesky of the packed P at `ps` into `lf` (both in this instance's record); every lane of the
// group factors redundantly in registers, lane 0 of the group publishes.  Returns pivot success.
template <int N>
SLB_DEV bool group_chol(const double *ps, double *lf, int sub) {
    constexpr int NP = N * (N + 1) / 2;
    double A[NP];
#pragma unroll
    for (int e = 0; e < NP; ++e) A[e] = ps[e];
    const bool ok = chol_packed_fast<N>(A);
    if (sub == 0) {
#pragma unroll
        for (int e = 0; e < NP; ++e) lf[e] = A[e];
    }
    __syncwarp();
    return ok;
}

// column j of the factor scaled by sgn (zero above the diagonal); s = 0 gives the zero vector
template <int N>
SLB_DEV void sigma_offset(const double *lf, int s, double *d) {
    const int j = s >= 1 ? (s - 1) >> 1 : 0;
    const double sgn = (s & 1) ? 1.0 : -1.0;
#pragma unroll
    for (int r = 0; r < N; ++r) d[r] = (s >= 1 && r >= j) ? sgn * lf[tri(r, j)] : 0.0;
}

// Msckf.hpp:471-496 / Usckf.hpp:601-627: reference = X0; do { d = mean(Xi [-] ref); ref [+]= d }
// while (|d| > 1e-6 && ++i < 10000).  Sigma points in `sig` as Y[c*NS + s].  `go` = this group takes
// part; groups of a warp that finish early idle through the remaining rounds.  Returns false when the
// iteration cap was hit.
template <class L, int G>
SLB_DEV bool group_mean(const double *sig, int sub, bool go, double *ref) {
    constexpr int N = L::N, QD = L::QD, NS = 2 * N + 1, ROUNDS = (NS + G - 1) / G;
#pragma unroll
    for (int c = 0; c < QD; ++c) ref[c] = sig[c * NS];
    int it = 0;
    while (__any_sync(FULL, go)) {
        double md[N];
#pragma unroll
        for (int r = 0; r < N; ++r) md[r] = 0.0;
#pragma unroll 2
        for (int t = 0; t < ROUNDS; ++t) {
            const int s = sub + G * t;
            if (s < NS) {
                double y[QD], d[N];
#pragma unroll
                for (int c = 0; c < QD; ++c) y[c] = sig[c * NS + s];
                boxminus<L>(y, ref, d);
#pragma unroll
                for (int r = 0; r < N; ++r) md[r] += d[r];
            }
        }
        double nrm2 = 0.0;
#pragma unroll
        for (int r = 0; r < N; ++r) {
            md[r] = gsum<G>(md[r]) * (1.0 / (double)NS);  // not "/ NS": zero numerators take div.rn's slow path
            nrm2 += md[r] * md[r];
        }
        double nr[QD];
        boxplus<L>(ref, md, 1.0, nr);
        if (go) {
#pragma unroll
            for (int c = 0; c < QD; ++c) ref[c] = nr[c];
            if (sqrt(nrm2) > 1e-6) {
                ++it;
                go = it < 10000;
            } else {
                go = false;
            }
        }
    }
    return it < 10000;
}

// Msckf.hpp:554-570: P = 0.5 * sum (Yi [-] mean)(Yi [-] mean)^T (+ Q), packed lower, written to `ps`.
// `sig` is consumed: it becomes the reduction scratch.  Q is the warp's packed shared Qp, or (QREG, per-instance noise)
// the entries e = sub + G k of this instance's packed Q, held in registers as Qp[k].
template <class L, int G, bool ADDQ, bool QREG = false>
SLB_DEV void group_cov(double *sig, double *ps, const double *Qp, int sub, const double *mean) {
    constexpr int N = L::N, QD = L::QD, NP = L::NP, NS = 2 * N + 1, ROUNDS = (NS + G - 1) / G;
    double acc[NP];
#pragma unroll
    for (int e = 0; e < NP; ++e) acc[e] = 0.0;
#pragma unroll 1
    for (int t = 0; t < ROUNDS; ++t) {
        const int s = sub + G * t;
        if (s < NS) {
            double y[QD], d[N];
#pragma unroll
            for (int c = 0; c < QD; ++c) y[c] = sig[c * NS + s];
            boxminus<L>(y, mean, d);
#pragma unroll
            for (int i = 0; i < N; ++i)
#pragma unroll
                for (int j = 0; j <= i; ++j) acc[tri(i, j)] = fma(d[i], d[j], acc[tri(i, j)]);
        }
    }
    __syncwarp();  // every lane is done with the sigma points: the area becomes scratch
#pragma unroll
    for (int e = 0; e < NP; ++e) sig[sub * NP + e] = acc[e];
    __syncwarp();
    if constexpr (QREG) {
#pragma unroll
        for (int k = 0; k < (NP + G - 1) / G; ++k) {
            const int e = sub + G * k;
            if (e < NP) {
                double v = sig[e];
#pragma unroll
                for (int l = 1; l < G; ++l) v += sig[l * NP + e];
                v *= 0.5;
                if (ADDQ) v += Qp[k];
                ps[e] = v;
            }
        }
    } else {
        for (int e = sub; e < NP; e += G) {
            double v = sig[e];
#pragma unroll
            for (int l = 1; l < G; ++l) v += sig[l * NP + e];
            v *= 0.5;
            if (ADDQ) v += Qp[e];
            ps[e] = v;
        }
    }
    __syncwarp();
}

// PIN: per-instance noise (slb_set_noise_layout).  Q and R are read at a.Q + inst * a.qs and a.R + inst * a.rs (a stride
// of 0 = shared).  Each 4-lane group fetches the entries of its own instance that it adds into registers -- lane sub the
// packed Q entries sub + 4k once the sigma points are drawn (the manifold-mean iterations cover their latency), every
// lane the 6 lower entries of R as the update starts; the warp's shared Qp is not used (8 per-instance copies per warp
// would cost a CTA).  Issued together with the record's copies they kept 18 more registers live through the predict and
// the fused MTK9 step spilled 264 / 308 B instead of 216 / 260 B.
// NIS: lane sub == 0 of each group stores the m2 its gate is given to a.nis[inst], NaN when the update's factorisation
// of P (or the predict before it) failed.
template <class L, int PM, class MM, int G, int TPB, int MINB, bool PRED, bool UPD, bool PIN = false, bool NIS = false>
__global__ void __launch_bounds__(TPB, MINB) ukf_kernel(slb::FilterArgs a) {
    typedef Rec<L, MM::M, G> R;
    constexpr int N = L::N, QD = L::QD, NP = L::NP, NS = 2 * N + 1, M = MM::M, MP = M * (M + 1) / 2;
    constexpr int IPW = 32 / G, WPB = TPB / 32, ROUNDS = (NS + G - 1) / G, RROWS = (N + G - 1) / G;
    constexpr int WSZ = UkfWarp<L, MM::M, G>::DOUBLES;  // per-warp shared memory: IPW records + packed Q + barrier
    static_assert(M == 3, "only 3-dof measurement models are wired to the UKF kernel");
    extern __shared__ double sm[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int sub = lane % G, grp = lane / G;
    double *wsm = sm + (size_t)warp * WSZ;
    double *rec = wsm + grp * R::IS;
    double *Qp = wsm + IPW * R::IS;
    uint64_t *ubar = reinterpret_cast<uint64_t *>(wsm + WSZ - 2);
    const int wbase = (blockIdx.x * WPB + warp) * IPW;  // first instance of this warp
    if (wbase >= a.B) return;
    const int inst = wbase + grp;
    const bool valid = inst < a.B;
    constexpr int QK = (NP + G - 1) / G;
    double qreg[PIN ? QK : 1], rreg[PIN ? MP : 1];   // PIN: this instance's noise (see above)
    const size_t ni = valid ? (size_t)inst : (size_t)(a.B - 1);   // idle tail groups borrow a real instance's noise

    // ---- stage the 8 records of this warp: lane -> (instance lane % IPW, fields lane / IPW + G k) ----
    // 8-byte LDGSTS: all ~14 loads of a lane are in flight before the first one lands (the staging loop used to
    // wait for each load in turn: 20 % of the kernel's stall samples)
    {
        const int li = lane % IPW, e0 = lane / IPW;
        const bool lv = wbase + li < a.B;
        double *dst = wsm + li * R::IS;
#pragma unroll 4
        for (int e = e0; e < QD + NP; e += G) {
            double *d = dst + (e < QD ? R::MU + e : R::PS + (e - QD));
            if (lv) {
                const double *src = e < QD ? a.mu + (size_t)e * a.stride + wbase + li : a.P + (size_t)(e - QD) * a.stride + wbase + li;
                cp_async8(d, src);
            } else {
                *d = 0.0;
            }
        }
        // u and z ride along: when they live in mapped host memory (zero-copy *_step_host) their PCIe latency is paid
        // once, together with the record's, instead of twice in the middle of the step.  A warp's 8 instances are one
        // contiguous run of each array (384 B of u, 192 B of z), fetched with ONE TMA bulk copy per array: over PCIe
        // that is a few large read requests instead of 18 sector-sized ones (the read-tag pool, not the link, bounded
        // the zero-copy step at ~23 GB/s).  They land in record 0's (not yet live) sigma-point area as u[8][NU] | z[8][M].
        {
            constexpr int NU = ProcessModel<PM>::NU, PERI = NU + M;
            static_assert(NU <= 6 && (IPW * NU * 8) % 16 == 0 && (IPW * M * 8) % 16 == 0, "bulk copy granularity");
            static_assert(IPW * PERI <= R::SIGSZ, "staging area");
            if (wbase + IPW <= a.B) {
                if (lane == 0) {
                    mbar_init(ubar, 1);
                    mbar_expect_tx(ubar, (PRED ? IPW * NU * 8 : 0) + (UPD ? IPW * M * 8 : 0));
                    if (PRED) bulk_g2s(wsm, a.u + (size_t)wbase * NU, IPW * NU * 8, ubar);
                    if (UPD) bulk_g2s(wsm + IPW * NU, a.z + (size_t)wbase * M, IPW * M * 8, ubar);
                }
            } else {   // ragged tail of the batch: element-wise
                for (int e = lane; e < IPW * PERI; e += 32) {
                    const int li2 = e / PERI, c = e - li2 * PERI;
                    double *d = c < NU ? wsm + li2 * NU + c : wsm + IPW * NU + li2 * M + (c - NU);
                    const bool need = c < NU ? PRED : UPD;
                    if (need && wbase + li2 < a.B) {
                        const double *src = c < NU ? a.u + (size_t)(wbase + li2) * NU + c : a.z + (size_t)(wbase + li2) * M + (c - NU);
                        cp_async8(d, src);
                    } else {
                        *d = 0.0;
                    }
                }
            }
        }
        if (PRED && !PIN) {
            for (int e = lane; e < NP; e += 32) {
                int r = (int)((sqrtf(8.0f * e + 1.0f) - 1.0f) * 0.5f);  // packed index -> (r, c), exact for e < 2^20
                r += (tri(r + 1, 0) <= e) - (tri(r, 0) > e);
                Qp[e] = __ldg(a.Q + r * N + (e - tri(r, 0)));
            }
        }
        cp_async_wait_all();
    }
    __syncwarp();
    if (wbase + IPW <= a.B) mbar_wait(ubar, 0);
    double *sig = rec + R::SIG, *lf = rec + R::LF, *ps = rec + R::PS;
    double ureg[ProcessModel<PM>::NU], zreg[MM::M];
#pragma unroll
    for (int c = 0; c < ProcessModel<PM>::NU; ++c) ureg[c] = PRED ? wsm[grp * ProcessModel<PM>::NU + c] : 0.0;
#pragma unroll
    for (int c = 0; c < MM::M; ++c) zreg[c] = UPD ? wsm[IPW * ProcessModel<PM>::NU + grp * MM::M + c] : 0.0;
    __syncwarp();
    if (!valid && sub == 0) {  // tail of the batch: a benign identity prior keeps the idle lanes finite
#pragma unroll
        for (int r = 0; r < N; ++r) ps[tri(r, r)] = 1.0;
#pragma unroll
        for (int b = 0; b < L::NB; ++b)
            if (L::so3(b)) rec[R::MU + L::qoff(b)] = 1.0;
    }
    __syncwarp();
    double mu[QD];
#pragma unroll
    for (int c = 0; c < QD; ++c) mu[c] = rec[R::MU + c];
    int st = 0;
    bool alive = valid;

    if (PRED) {
        // ---- predict(g, Q): sigma points -> g -> manifold mean -> cov + Q ------------------------
        if (!group_chol<N>(ps, lf, sub) && alive) { st |= SLB_ST_CHOL_FAIL; alive = false; }
        ProcessModel<PM> g;
        {
            double u[ProcessModel<PM>::NU];
#pragma unroll
            for (int c = 0; c < ProcessModel<PM>::NU; ++c) u[c] = ureg[c];
            g.prepare(u, a.dt);
        }
#pragma unroll 1
        for (int t = 0; t < ROUNDS; ++t) {
            const int s = sub + G * t;
            if (s < NS) {
                double d[N], x[QD], y[QD];
                sigma_offset<N>(lf, s, d);
                boxplus<L>(mu, d, 1.0, x);
                g.apply(x, y);
#pragma unroll
                for (int c = 0; c < QD; ++c) sig[c * NS + s] = y[c];
            }
        }
        if (PIN) {
            const double *Qi = a.Q + ni * a.qs;
#pragma unroll
            for (int k = 0; k < QK; ++k) {
                const int e = sub + G * k;
                int r = (int)((sqrtf(8.0f * e + 1.0f) - 1.0f) * 0.5f);
                r += (tri(r + 1, 0) <= e) - (tri(r, 0) > e);
                qreg[k] = e < NP ? __ldg(Qi + r * N + (e - tri(r, 0))) : 0.0;
            }
        }
        __syncwarp();
        if (!group_mean<L, G>(sig, sub, alive, mu) && alive) st |= SLB_ST_MEAN_NOCONV;
        if constexpr (PIN) group_cov<L, G, true, true>(sig, ps, qreg, sub, mu);
        else group_cov<L, G, true>(sig, ps, Qp, sub, mu);
    }

    if (UPD) {
        // ---- update(z, h, R, mt) ----------------------------------------------------------------
        // `alive` = the record holds something to publish (in the fused step: the predicted state); a failing update
        // leaves that state as it is, exactly like calling predict and update separately
        bool upd = alive;
        if (PIN) {
            const double *Ri = a.R + ni * a.rs;
#pragma unroll
            for (int r = 0; r < M; ++r)
#pragma unroll
                for (int c = 0; c <= r; ++c) rreg[tri(r, c)] = __ldg(Ri + r * M + c);
        }
        if (!group_chol<N>(ps, lf, sub) && alive) { st |= SLB_ST_CHOL_FAIL; upd = false; }
        double *Z = sig + R::ZO, *DZ = sig + R::DZO, *Ks = sig + R::KO, *KSs = sig + R::KSO, *DL = sig + R::DLO;
        double zsum[M];
#pragma unroll
        for (int c = 0; c < M; ++c) zsum[c] = 0.0;
#pragma unroll 1
        for (int t = 0; t < ROUNDS; ++t) {
            const int s = sub + G * t;
            if (s < NS) {
                double d[N], x[QD], z[M];
                sigma_offset<N>(lf, s, d);
                boxplus<L>(mu, d, 1.0, x);
                MM::apply(x, z);
#pragma unroll
                for (int c = 0; c < M; ++c) { Z[c * NS + s] = z[c]; zsum[c] += z[c]; }
            }
        }
        double zbar[M];
#pragma unroll
        for (int c = 0; c < M; ++c) zbar[c] = gsum<G>(zsum[c]) * (1.0 / (double)NS);
        __syncwarp();
        // S = 0.5 sum (Zi - zbar)(Zi - zbar)^T + R   (packed lower)
        double S[MP];
#pragma unroll
        for (int e = 0; e < MP; ++e) S[e] = 0.0;
#pragma unroll 1
        for (int t = 0; t < ROUNDS; ++t) {
            const int s = sub + G * t;
            if (s < NS) {
                double dz[M];
#pragma unroll
                for (int c = 0; c < M; ++c) dz[c] = Z[c * NS + s] - zbar[c];
#pragma unroll
                for (int r = 0; r < M; ++r)
#pragma unroll
                    for (int c = 0; c <= r; ++c) S[tri(r, c)] += dz[r] * dz[c];
            }
        }
#pragma unroll
        for (int r = 0; r < M; ++r)
#pragma unroll
            for (int c = 0; c <= r; ++c) S[tri(r, c)] = 0.5 * gsum<G>(S[tri(r, c)]) + (PIN ? rreg[tri(r, c)] : __ldg(a.R + r * M + c));
        // Pxz = 0.5 sum (Xi [-] mu)(Zi - zbar)^T.  Xi [-] mu is +-L e_j by construction (the reference
        // recovers it through log(exp(.)), identical below |.| < pi), and the zbar terms of a +- pair
        // cancel: Pxz = 0.5 L DZ with DZ_j = Z+_j - Z-_j.
        for (int j = sub; j < N; j += G) {
#pragma unroll
            for (int c = 0; c < M; ++c) DZ[j * M + c] = (Z[c * NS + 1 + 2 * j] - zbar[c]) - (Z[c * NS + 2 + 2 * j] - zbar[c]);
        }
        __syncwarp();
        double Si[MP];
        sym3_inverse(S, Si);
        auto SiAt = [&](int r, int c) { return r >= c ? Si[tri(r, c)] : Si[tri(c, r)]; };
        auto SAt = [&](int r, int c) { return r >= c ? S[tri(r, c)] : S[tri(c, r)]; };
        double innov[M], m2 = 0.0;
#pragma unroll
        for (int c = 0; c < M; ++c) innov[c] = zreg[c] - zbar[c];
#pragma unroll
        for (int r = 0; r < M; ++r) {
            double s = 0.0;
#pragma unroll
            for (int c = 0; c < M; ++c) s += SiAt(r, c) * innov[c];
            m2 += innov[r] * s;
        }
        // rows sub, sub+G, ... of Pxz, K = Pxz S^-1, K S and delta = K innovation
#pragma unroll
        for (int t = 0; t < RROWS; ++t) {
            const int r = sub + G * t;
            if (r < N) {
                double px[M];
#pragma unroll
                for (int c = 0; c < M; ++c) px[c] = 0.0;
                for (int j = 0; j <= r; ++j) {
                    const double l = lf[tri(r, j)];
#pragma unroll
                    for (int c = 0; c < M; ++c) px[c] = fma(l, DZ[j * M + c], px[c]);
                }
                double K[M], dsum = 0.0;
#pragma unroll
                for (int c = 0; c < M; ++c) {
                    double s = 0.0;
#pragma unroll
                    for (int p = 0; p < M; ++p) s += (0.5 * px[p]) * SiAt(p, c);
                    K[c] = s;
                    dsum += s * innov[c];
                }
#pragma unroll
                for (int c = 0; c < M; ++c) {
                    double s = 0.0;
#pragma unroll
                    for (int p = 0; p < M; ++p) s += K[p] * SAt(p, c);
                    Ks[r * M + c] = K[c];
                    KSs[r * M + c] = s;
                }
                DL[r] = dsum;
            }
        }
        __syncwarp();
        if (NIS && sub == 0 && valid) a.nis[inst] = upd ? m2 : __longlong_as_double(0x7ff8000000000000ll);
        const bool accept = chi2_accept(m2, a.gate);
        if (upd && !accept) st |= SLB_ST_GATE_REJECT;
        const bool apply = upd && accept;
        // the prior covariance of this update, kept until the update is known to go through
        double Psave[(NP + G - 1) / G];
#pragma unroll
        for (int k = 0; k < (NP + G - 1) / G; ++k) Psave[k] = (sub + G * k < NP) ? ps[sub + G * k] : 0.0;
        __syncwarp();
        // sigma -= K S K^T   (lower triangle; the reference's LLT reads only that, Q8)
        if (apply) {
#pragma unroll
            for (int t = 0; t < RROWS; ++t) {
                const int r = sub + G * t;
                if (r < N) {
                    const double k0 = KSs[r * M], k1 = KSs[r * M + 1], k2 = KSs[r * M + 2];
                    for (int c = 0; c <= r; ++c)
                        ps[tri(r, c)] -= k0 * Ks[c * M] + k1 * Ks[c * M + 1] + k2 * Ks[c * M + 2];
                }
            }
        }
        double delta[N];
#pragma unroll
        for (int r = 0; r < N; ++r) delta[r] = DL[r];
        __syncwarp();
        // apply_delta(K * innovation): re-draw sigma points around mu [+] delta.  Groups that do not
        // apply (gate, earlier failure) run the same instructions on their untouched P and drop the result.
        if (!apply) {
#pragma unroll
            for (int r = 0; r < N; ++r) delta[r] = 0.0;
        }
        const bool ok3 = group_chol<N>(ps, lf, sub);
        if (apply && !ok3) st |= SLB_ST_CHOL_FAIL;
        const bool done = apply && ok3;
#pragma unroll 1
        for (int t = 0; t < ROUNDS; ++t) {
            const int s = sub + G * t;
            if (s < NS) {
                double d[N], x[QD];
                sigma_offset<N>(lf, s, d);
#pragma unroll
                for (int r = 0; r < N; ++r) d[r] += delta[r];
                boxplus<L>(mu, d, 1.0, x);
#pragma unroll
                for (int c = 0; c < QD; ++c) sig[c * NS + s] = x[c];
            }
        }
        __syncwarp();
        double nm[QD];
        const bool conv = group_mean<L, G>(sig, sub, done, nm);
        if (done) {
            if (!conv) st |= SLB_ST_MEAN_NOCONV;
#pragma unroll
            for (int c = 0; c < QD; ++c) mu[c] = nm[c];
        }
        group_cov<L, G, false>(sig, ps, Qp, sub, nm);
        if (!done) {  // rejected / failed update: sigma and mu stay as they were (Usckf.hpp:294 / ukf::update)
#pragma unroll
            for (int k = 0; k < (NP + G - 1) / G; ++k)
                if (sub + G * k < NP) ps[sub + G * k] = Psave[k];
        }
    }

    // ---- publish: mean to the record, status, then the warp streams its records back to HBM ---------
    bool finite = true;
#pragma unroll
    for (int c = 0; c < QD; ++c) finite = finite && isfinite(mu[c]);
    if (alive && !finite) st |= SLB_ST_NONFINITE;
    if (sub == 0) {
#pragma unroll
        for (int c = 0; c < QD; ++c) rec[R::MU + c] = mu[c];
        rec[R::FLAG] = alive ? 1.0 : 0.0;
        if (st && valid) a.status[inst] |= st;
    }
    __syncwarp();
    {
        const int li = lane % IPW, e0 = lane / IPW;
        const double *src = wsm + li * R::IS;
        if (wbase + li < a.B && src[R::FLAG] != 0.0) {
#pragma unroll 4
            for (int e = e0; e < QD + NP; e += G) {
                if (e < QD) a.mu[(size_t)e * a.stride + wbase + li] = src[R::MU + e];
                else a.P[(size_t)(e - QD) * a.stride + wbase + li] = src[R::PS + (e - QD)];
            }
        }
    }
    // Optional instance-major copy of the posterior means (the *_step_host entry points pass mapped host memory here:
    // the warp's 8 q-vectors are 640 contiguous bytes, written with full-width coalesced stores straight over PCIe).
    if (a.mu_out) {
        const int OL = a.out_len;
        for (int e = lane; e < IPW * OL; e += 32) {
            const int li = e / OL, c = a.out_off + (e - li * OL);
            if (wbase + li < a.B) {
                const double *src = wsm + li * R::IS;
                // a failed instance keeps its prior, which is what the state arrays still hold
                a.mu_out[(size_t)(wbase + li) * OL + (c - a.out_off)] =
                    src[R::FLAG] != 0.0 ? src[R::MU + c] : a.mu[(size_t)c * a.stride + wbase + li];
            }
        }
    }
}

}  // namespace slbd

namespace slb {

// Per-instance noise (a.qs / a.rs set by slb_set_noise_layout) selects the PIN instantiations, NIS capture (a.nis) the
// NIS ones of the update-bearing kernels; the shared-noise kernels are unchanged.
template <class L, int PM, class MM>
static int launch_ukf_t(bool predict, bool update, const FilterArgs &a, cudaStream_t s) {
    constexpr int G = 4, TPB = 128, MINB = 3;
    typedef slbd::Rec<L, MM::M, G> R;
    constexpr size_t smem = (size_t)(TPB / 32) * slbd::UkfWarp<L, MM::M, G>::DOUBLES * sizeof(double);
    static_assert(smem <= 227 * 1024, "instance records exceed shared memory");
    const int ipb = TPB / G;
    const int grid = (a.B + ipb - 1) / ipb;
    auto go = [&](auto kern) -> int {
        SLB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        kern<<<grid, TPB, smem, s>>>(a);
        count_launch();
        SLB_CUDA(cudaGetLastError());
        return SLB_OK;
    };
    const bool pin = (predict && a.qs) || (update && a.rs);
    if (update && a.nis) {
        if (pin) return predict ? go(slbd::ukf_kernel<L, PM, MM, G, TPB, MINB, true, true, true, true>)
                                : go(slbd::ukf_kernel<L, PM, MM, G, TPB, MINB, false, true, true, true>);
        return predict ? go(slbd::ukf_kernel<L, PM, MM, G, TPB, MINB, true, true, false, true>)
                       : go(slbd::ukf_kernel<L, PM, MM, G, TPB, MINB, false, true, false, true>);
    }
    if (pin) {
        if (predict && update) return go(slbd::ukf_kernel<L, PM, MM, G, TPB, MINB, true, true, true>);
        if (predict) return go(slbd::ukf_kernel<L, PM, MM, G, TPB, MINB, true, false, true>);
        if (update) return go(slbd::ukf_kernel<L, PM, MM, G, TPB, MINB, false, true, true>);
    }
    if (predict && update) return go(slbd::ukf_kernel<L, PM, MM, G, TPB, MINB, true, true>);
    if (predict) return go(slbd::ukf_kernel<L, PM, MM, G, TPB, MINB, true, false>);
    if (update) return go(slbd::ukf_kernel<L, PM, MM, G, TPB, MINB, false, true>);
    return set_error(SLB_ERR_INVALID, "ukf: nothing to do");
}

int launch_ukf(int layout, int pm, int mm, bool predict, bool update, const FilterArgs &a, cudaStream_t s) {
    using namespace slbd;
    if (update && mm != SLB_MM_GPS_POS) return set_error(SLB_ERR_INVALID, "ukf: unsupported measurement model");
    if (!predict) pm = layout == SLB_LAYOUT_POSE6 ? SLB_PM_POSE6_ODOM : SLB_PM_UKFOM_IMU;
    if (layout == SLB_LAYOUT_MTK9 && pm == SLB_PM_UKFOM_IMU)
        return launch_ukf_t<LayMtk9, SLB_PM_UKFOM_IMU, MmGpsPos>(predict, update, a, s);
    if (layout == SLB_LAYOUT_MTK9 && pm == SLB_PM_UKFOM_IMU_REFBUG)
        return launch_ukf_t<LayMtk9, SLB_PM_UKFOM_IMU_REFBUG, MmGpsPos>(predict, update, a, s);
    if (layout == SLB_LAYOUT_POSE6 && pm == SLB_PM_POSE6_ODOM)
        return launch_ukf_t<LayPose6, SLB_PM_POSE6_ODOM, MmGpsPos>(predict, update, a, s);
    return set_error(SLB_ERR_INVALID, "ukf: unsupported layout / process model combination");
}

}  // namespace slb
