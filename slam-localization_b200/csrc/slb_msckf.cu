// slb_msckf.cu -- localization::Msckf<MultiState<State,SensorState>,State> (src/filters/Msckf.hpp):
// predict (warp per instance, shared with the USCKF predict) and the UKF-flavoured update with the
// per-feature chi-square gate, one filter instance per CTA.
//
// update (Msckf.hpp:220-277, removeOutliers :723-754, applyDelta :659-666) at BASELINE config 3
// (10 clones -> N = 72, 145 sigma points, 50 features -> m = 100) keeps everything of one instance in
// shared memory (~224 KB: one CTA per SM, persistent over the batch):
//   A  5056 doubles : P -> L (Cholesky in place) ... later S -> Ls ... later P_new -> L2
//   B 14800 doubles : Z (148 x 100) ... later compacted S' (outliers) ... later X / D (148 x 84)
//   C  7200 doubles : W -> covXZ (in-place TRMM) -> Y = covXZ Ls^-T (in place, inside chol_blocked)
// Algebra: with S = Ls Ls^T and Y = covXZ Ls^-T the reference's  K = covXZ S^-1, Pk -= K S K^T,
// delta = K nu  become  Pk -= Y Y^T,  delta = Y (Ls^-1 nu)  -- same maths as :257-263 without forming
// the explicit inverse (quirk Q9).  covXZ = L W with W_j = 0.5 (Z+_j - Z-_j), as in the other kernels.
//
// FP64 tensor cores: every rank-k contraction here (S = Zc^T Zc, covXZ = L W, the trailing updates of the
// blocked Cholesky / triangular solve, P - Y Y^T, the re-estimated covariance D^T D) runs as 8x8x4 DMMA
// tiles (m8n8k4, dmma884).  profiles/r01_dmma_vs_dfma_peak.txt: on B200 the DMMA pipe delivers the same
// 37 TFLOP/s as the SIMT FP64 pipe, so it does not raise the roofline -- but one DMMA replaces 8 DFMA issue
// slots per lane and needs 2 operand loads per 8 FMA instead of the 4x4 register tile's 8 per 16, and this
// kernel was bound by instruction issue and shared-memory operand traffic (FP64 pipe 7.5 % busy before),
// not by FP64 throughput.  Row strides of the [k][col] / [row][k] operand arrays are = 4 (mod 16) doubles so a
// fragment load (4 k x 8 rows-or-cols) touches 32 distinct banks.
#include "slb_predict12.cuh"

namespace slbd {

constexpr int MS_T = 512;          // threads per CTA (16 warps: 126 registers, no spills; 256 -> 512 gave +10..13 %, 768 spills)
constexpr int MS_W = MS_T / 32;
constexpr int MS_NMAX = 72, MS_MMAX = 100, MS_NSMAX = 145;
constexpr int MS_NSPAD = 148;                    // sigma-point count padded to the DMMA k-step
static_assert(MS_NSMAX == 2 * MS_NMAX + 1 && MS_NSPAD >= MS_NSMAX && MS_NSPAD % 4 == 0, "sigma-point padding");
constexpr int MS_A = 5056;                       // >= 100*101/2 and >= 72*73/2
constexpr int MS_ZS = 100;                       // row stride of Z and of covXZ / Y   (= 4 mod 16)
constexpr int MS_QS = 84;                        // q-vector scalars per sigma point (13 + 7 * 10, padded)
constexpr int MS_XS = MS_NSPAD;                  // the sigma points X / deviations D are stored TRANSPOSED, Xt[scalar][sigma point],
                                                 // row stride 148 (= 4 mod 16): a lane per sigma point reads consecutive doubles
                                                 // (the [sigma point][scalar] layout made those accesses 8-way bank conflicts) and
                                                 // the DMMA fragments of D^T D (4 sigma points x 8 scalars) still hit 32 banks
constexpr int MS_B = MS_NSPAD * MS_ZS;           // 14800
constexpr int MS_C = MS_NMAX * MS_ZS;            // 7200
constexpr int MS_D = 896;                        // small vectors
constexpr int MS_SMEM_DOUBLES = MS_A + MS_B + MS_C + MS_D;
static_assert(MS_SMEM_DOUBLES * 8 <= 227 * 1024, "MSCKF update working set exceeds shared memory");
static_assert(MS_QS * MS_XS <= MS_B && MS_XS % 16 == 4, "sigma points do not fit region B");
static_assert(MS_MMAX * (MS_MMAX + 1) / 2 <= MS_A && MS_A + 2 * 1600 <= MS_B, "compacted S + two panel stagings do not fit region B");
static_assert(2400 >= 32 * MS_NMAX && 2400 + MS_NMAX * (MS_NMAX + 1) / 2 <= MS_C, "parked factor does not fit region C");

// linear index of a lower-triangular tile -> (tr, tc), tc <= tr: a constant-memory table (the index is warp-uniform,
// so the lookup is one broadcast load instead of a sqrtf + fix-up per tile)
struct TileTab {
    unsigned char tr[128], tc[128];   // 13 tile rows (m = 100) need 91 entries
    constexpr TileTab() : tr(), tc() {
        int r = 0, c = 0;
        for (int t = 0; t < 128; ++t) {
            tr[t] = (unsigned char)r;
            tc[t] = (unsigned char)c;
            if (++c > r) { c = 0; ++r; }
        }
    }
};
__constant__ TileTab tile_tab = TileTab();
static_assert((MS_MMAX + 7) / 8 * ((MS_MMAX + 7) / 8 + 1) / 2 <= 128, "tile table too small");
SLB_DEV void tri_tile(int t, int &tr, int &tc) {
    tr = tile_tab.tr[t];
    tc = tile_tab.tc[t];
}

// In-place Cholesky of a packed lower matrix in shared memory, all threads of the CTA.  Blocked right-looking
// with 8-wide panels: warp 0 factors the 8x8 diagonal block (lane per row, shuffle broadcasts), one thread per
// row solves the panel below it, then the other warps rank-8-update the trailing 8x8 tiles with two DMMAs each
// while warp 0 already factors the next diagonal block (look-ahead).  invd[i] = 1 / L_ii is left for later
// triangular solves.  ok_flag (shared int) is cleared on a non-positive pivot (Eigen::LLT's info(), which the
// reference ignores: quirk Q8).
// Optional right-hand sides: nx rows X (row stride xs) plus one more row xe are carried through the same panel
// solves and trailing updates, i.e. on return [X; xe] holds [X; xe] L^-T -- the triangular solve a Cholesky is
// usually followed by, without its own serial panel chain and barriers.
// Optional inverse factor: Wp (packed lower) receives L^-1.  It is the right-hand side I carried through the factorisation,
// stored transposed -- row i of the right-hand side is column i of Wp -- so that I L^-T lands as its transpose.  Only the
// tiles that can be non-zero (row tile <= current panel) exist; nothing has to be preset.
// PS is a 1600-double scratch: every solved panel is also parked there as dense 8-wide rows, swizzled so that the
// DMMA fragment loads of the trailing update are bank-conflict free (the packed triangle's row starts are not:
// 2.4 wavefronts per ideal one, and the tiles are shared-memory-bandwidth bound).
// -DSLB_CHOL_TIMING=<call index>: per-panel clock64() stamps of one chol_blocked call of CTA 0 (profiles/chol_timing.py)
#ifdef SLB_CHOL_TIMING
__device__ long long chol_dbg[16 * 16 * 8];   // [panel][warp][slot]
__device__ int chol_dbg_call;
#define CHOL_T(panel, slot) do { if (blockIdx.x == 0 && chol_dbg_call == SLB_CHOL_TIMING && (threadIdx.x & 31) == 0 && (panel) < 16) chol_dbg[((panel) * 16 + (threadIdx.x >> 5)) * 8 + (slot)] = clock64(); } while (0)
#else
#define CHOL_T(panel, slot) do { } while (0)
#endif
// -DSLB_MSCKF_PHASES: clock64() stamp of thread 0 of CTA 0 at every phase boundary of msckf_update_kernel, for its
// second and third instance (steady state: the factor of P arrives from the previous iteration) -- profiles/msckf_phases.py
#ifdef SLB_MSCKF_PHASES
__device__ long long ms_phase_dbg[4 * 32];
#define MS_PH(slot) do { if (blockIdx.x == 0 && threadIdx.x == 0 && ms_it < 4) ms_phase_dbg[ms_it * 32 + (slot)] = clock64(); } while (0)
#else
#define MS_PH(slot) do { } while (0)
#endif
constexpr int MS_PS = 1600;
constexpr int MS_NXL = 2400;   // offset in region C of the next instance's factor (above the <= 32 x 72 partial sums of the mean)
SLB_DEV int ps_idx(int srow, int k) { return srow * 8 + ((k + 4 * ((srow >> 1) & 1)) & 7); }
SLB_DEV void chol_blocked(double *A, int n, int *ok_flag, double *invd, double *PS, double *X = nullptr, int nx = 0,
                          int xs = 0, double *xe = nullptr, double *Wp = nullptr) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int fr = lane >> 2, fk = lane & 3;
    const int nxr = X ? nx + 1 : 0, nxt = (nxr + 7) >> 3;
    // inverse of a diagonal block, row-major 8 x 8, double-buffered by panel parity: the look-ahead writes the next panel's
    // while the right-hand-side tasks still read the current one (staging uses < 184 of the 200 rows of PS)
    auto dinv_of = [&](int p0) { return PS + MS_PS - 128 + 64 * ((p0 >> 3) & 1); };
    // 8x8 diagonal block on one warp, two entries per lane in the DMMA accumulator layout (row fr, columns 2 fk and
    // 2 fk + 1).  Right-looking and square-root-free: step k broadcasts d_k = a_kk, a_ik and a_jk by shuffles, then
    // a_ij -= (a_ik / d_k) a_jk is ONE FMA per entry -- the dependent chain per column is shuffle + reciprocal + multiply +
    // FMA and there is hardly any other instruction to issue (lane-per-row needed up to 7 shuffle + FMA pairs per step).
    // The same Gauss transforms are accumulated on the identity (M = prod (I - v_k e_k^T)): diag(1 / L_ii) M is the inverse
    // of the block, which turns the panel solve below it from an 8-step forward substitution per row into 36 independent
    // FMAs per row.  All square roots are taken after the loop.
    auto factor_diag = [&](int p0, double a0, double a1) {   // a0, a1: this lane's two entries (0 outside the lower triangle)
        const int pb = min(8, n - p0);
        const int i = fr, j0 = 2 * fk, j1 = j0 + 1;
        double *dinv = dinv_of(p0);
        double m0 = (i == j0) ? 1.0 : 0.0, m1 = (i == j1) ? 1.0 : 0.0;
        double di = 1.0, dj0 = 1.0, dj1 = 1.0;   // pivots of this lane's row and of its two columns
        bool ok = true;
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            if (k < pb) {
                const int kh = k >> 1;
                const double ak = (k & 1) ? a1 : a0;                       // this lane's entry in column pair kh
                const double d = bcast(ak, 4 * k + kh);                    // a_kk
                const double aik = __shfl_sync(0xffffffffu, ak, 4 * i + kh);
                ok = ok && (d > 0.0);
                if (i == k) di = d;
                if (j0 == k) dj0 = d;
                if (j1 == k) dj1 = d;
                if (k < 7) {
                    const double ajk0 = __shfl_sync(0xffffffffu, ak, 4 * j0 + kh), ajk1 = __shfl_sync(0xffffffffu, ak, 4 * j1 + kh);
                    const double mk0 = bcast(m0, 4 * k + fk), mk1 = bcast(m1, 4 * k + fk);
                    const double v = aik * rcp_fast(d);
                    if (j0 > k) a0 = fma(-v, ajk0, a0);
                    if (j1 > k) a1 = fma(-v, ajk1, a1);
                    const double vm = i > k ? v : 0.0;
                    m0 = fma(-vm, mk0, m0);
                    m1 = fma(-vm, mk1, m1);
                }
            }
        }
        double si, ri, s0, r0c, s1, r1c;
        sqrt_rsqrt(di, si, ri);
        sqrt_rsqrt(dj0, s0, r0c);
        sqrt_rsqrt(dj1, s1, r1c);
        if (i < pb) {
            if (fk == 0) invd[p0 + i] = ri;
            if (j0 <= i) A[tri(p0 + i, p0 + j0)] = (j0 == i) ? s0 : a0 * r0c;
            if (j1 <= i) A[tri(p0 + i, p0 + j1)] = (j1 == i) ? s1 : a1 * r1c;
        }
        *reinterpret_cast<double2 *>(dinv + i * 8 + j0) = make_double2(j0 <= i ? ri * m0 : 0.0, j1 <= i ? ri * m1 : 0.0);
        ok = __all_sync(0xffffffffu, ok);
        if (!ok && lane == 0) *ok_flag = 0;
    };
    if (warp == 0) {
        const int pb = min(8, n);
        factor_diag(0, (fr < pb && 2 * fk <= fr) ? A[tri(fr, 2 * fk)] : 0.0, (fr < pb && 2 * fk + 1 <= fr) ? A[tri(fr, 2 * fk + 1)] : 0.0);
    }
    __syncthreads();
    for (int p0 = 0; p0 < n; p0 += 8) {
        const int pb = min(8, n - p0);
        const int r0 = p0 + pb, na = n - r0;
        const double *dinv = dinv_of(p0);
        CHOL_T(p0 >> 3, 0);
        // panel below the diagonal block: rows * inv(L_pp)^T, one 8-row tile per warp as two DMMAs (B[k][c] = Dinv[c][k]); the
        // result goes back in place and, as dense swizzled 8-wide rows, into the staging area for the fragment loads of the
        // trailing update.  na > 0 implies a full panel (pb == 8).
        for (int rt = warp; 8 * rt < na; rt += MS_W) {
            const int w = 8 * rt + fr, wc = min(w, na - 1);
            const double *Ai = A + tri(r0 + wc, p0);
            double x0 = 0.0, x1 = 0.0;
            dmma884(x0, x1, Ai[fk], dinv[fr * 8 + fk]);
            dmma884(x0, x1, Ai[fk + 4], dinv[fr * 8 + fk + 4]);
            __syncwarp();   // every lane has read its fragment of the rows before they are overwritten
            if (w < na) {
                double *Ao = A + tri(r0 + w, p0) + 2 * fk;
                Ao[0] = x0;
                Ao[1] = x1;
                *reinterpret_cast<double2 *>(PS + ps_idx(w, 2 * fk)) = make_double2(x0, x1);
            }
        }
        CHOL_T(p0 >> 3, 1);
        __syncthreads();
        CHOL_T(p0 >> 3, 2);
        // rows / columns beyond the matrix only feed accumulator entries that are never stored: their addresses are clamped,
        // not masked; a trailing update only exists after a full 8-wide panel (pb == 8), so the k-loop needs no bound either
        const int nt = (na + 7) >> 3, ntiles = nt * (nt + 1) / 2;
        // operands come from the staged panel; rows beyond the matrix are clamped (their accumulator rows are dropped)
        auto a_tile = [&](int t) {
            int tr, tc;
            tri_tile(t, tr, tc);
            const int i0 = r0 + 8 * tr, j0 = r0 + 8 * tc;
            double d0 = 0.0, d1 = 0.0;
            const int ra = min(8 * tr + fr, na - 1), rb = min(8 * tc + fr, na - 1);
            const int i = i0 + fr, j = j0 + 2 * fk;
            const bool v0 = i < n && j <= i, v1 = i < n && j + 1 <= i;
            double *po = A + tri(min(i, n - 1), min(j, i));   // old values requested together with the operands
            const double c0 = v0 ? po[0] : 0.0, c1 = v1 ? po[1] : 0.0;
            dmma884(d0, d1, PS[ps_idx(ra, fk)], PS[ps_idx(rb, fk)]);
            dmma884(d0, d1, PS[ps_idx(ra, fk + 4)], PS[ps_idx(rb, fk + 4)]);
            if (v0) po[0] = c0 - d0;
            if (v1) po[1] = c1 - d1;
        };
        if (warp == 0) {
            if (ntiles > 0) {
                // look-ahead: warp 0 owns the next diagonal block.  Its trailing update (both operands are the staged rows
                // 0..7) leaves the block in the accumulator layout, which is the layout factor_diag works in: no round trip
                // through shared memory; the factorisation runs while the other warps update their tiles.
                const int rr = min(fr, na - 1), pbn = min(8, na);
                const int i = r0 + fr, j = r0 + 2 * fk;
                const bool v0 = fr < pbn && 2 * fk <= fr, v1 = fr < pbn && 2 * fk + 1 <= fr;
                const double x0 = PS[ps_idx(rr, fk)], x1 = PS[ps_idx(rr, fk + 4)];
                const double c0 = v0 ? A[tri(i, j)] : 0.0, c1 = v1 ? A[tri(i, j + 1)] : 0.0;
                double d0 = 0.0, d1 = 0.0;
                dmma884(d0, d1, x0, x0);
                dmma884(d0, d1, x1, x1);
                CHOL_T(p0 >> 3, 3);
                factor_diag(r0, v0 ? c0 - d0 : 0.0, v1 ? c1 - d1 : 0.0);
            }
        } else {
            // Work list of the 15 other warps, longest tasks first:
            //   [0, nxq)        right-hand-side rows X, LEFT-looking: columns p0..p0+7 of 16 rows are finished here,
            //                   X(:, p) = (X(:, p) - sum_{q < p} X(:, q) L(p, q)^T) inv(L_pp)^T -- a register-accumulated k-loop
            //                   (one shared L fragment for two row tiles) instead of a read-modify-write of every trailing
            //                   tile at every panel; this work grows with p while the trailing tiles shrink
            //   [nxq, nxq+nwt)  identity right-hand side (Wp), left-looking in the same way; row tile r <= p starts its k-loop at
            //                   column 8r, and the diagonal tile r = p is inv(L_pp)^T itself
            //   then            trailing tiles 1.. of the matrix (right-looking, tile 0 is warp 0's)
            const int nwt = Wp ? (p0 >> 3) + 1 : 0;   // row tiles of the identity right-hand side reached so far
            const int nxq = (nxt + 1) >> 1, nat = max(ntiles - 1, 0);
            // warps 4, 8, 12 share warp 0's scheduler (and its FP64 pipe): they come last in the task order, so the long
            // right-hand-side tasks never land next to the diagonal factorisation
            const int rank = (warp & 3) ? (warp >> 2) * 3 + (warp & 3) - 1 : 11 + (warp >> 2);
            for (int t = rank; t < nxq + nwt + nat; t += MS_W - 1) {
                if (t < nxq) {
                    const int ia = 16 * t + fr, ib = ia + 8, ca = min(ia, nxr - 1), cb = min(ib, nxr - 1);
                    double *xa = ca < nx ? X + ca * xs : xe, *xb = cb < nx ? X + cb * xs : xe;
                    const double *lrow = A + tri(min(p0 + fr, n - 1), 0) + fk;   // L(p0 + fr, q + fk): B fragment
                    double d0 = 0.0, d1 = 0.0, e0 = 0.0, e1 = 0.0;
                    {   // p0 is a multiple of 8: two k-steps per trip on separate accumulators (four DMMA chains in flight)
                        double d2 = 0.0, d3 = 0.0, e2 = 0.0, e3 = 0.0;
#pragma unroll 2
                        for (int q = 0; q < p0; q += 8) {
                            const double bl0 = lrow[q], bl1 = lrow[q + 4];
                            const double xa0 = xa[q + fk], xa1 = xa[q + fk + 4], xb0 = xb[q + fk], xb1 = xb[q + fk + 4];
                            dmma884(d0, d1, xa0, bl0);
                            dmma884(e0, e1, xb0, bl0);
                            dmma884(d2, d3, xa1, bl1);
                            dmma884(e2, e3, xb1, bl1);
                        }
                        d0 += d2; d1 += d3; e0 += e2; e1 += e3;
                    }
                    const int c0 = p0 + 2 * fk, k0 = p0 + fk, k1 = k0 + 4;
                    const bool v0 = c0 < n, v1 = c0 + 1 < n, oka = ia < nxr, okb = ib < nxr;
                    // (X - sum) goes back in place so that it can be re-read as an A fragment for the product with inv(L_pp)^T
                    const double ta0 = (v0 ? xa[c0] : 0.0) - d0, ta1 = (v1 ? xa[c0 + 1] : 0.0) - d1;
                    const double tb0 = (v0 ? xb[c0] : 0.0) - e0, tb1 = (v1 ? xb[c0 + 1] : 0.0) - e1;
                    if (oka && v0) xa[c0] = ta0;
                    if (oka && v1) xa[c0 + 1] = ta1;
                    if (okb && v0) xb[c0] = tb0;
                    if (okb && v1) xb[c0 + 1] = tb1;
                    __syncwarp();
                    const double aa0 = k0 < n ? xa[k0] : 0.0, aa1 = k1 < n ? xa[k1] : 0.0;
                    const double ab0 = k0 < n ? xb[k0] : 0.0, ab1 = k1 < n ? xb[k1] : 0.0;
                    const double bd0 = dinv[fr * 8 + fk], bd1 = dinv[fr * 8 + fk + 4];   // B[k][c] = Dinv[c][k]
                    double f0 = 0.0, f1 = 0.0, g0 = 0.0, g1 = 0.0;
                    dmma884(f0, f1, aa0, bd0);
                    dmma884(g0, g1, ab0, bd0);
                    dmma884(f0, f1, aa1, bd1);
                    dmma884(g0, g1, ab1, bd1);
                    __syncwarp();
                    if (oka && v0) xa[c0] = f0;
                    if (oka && v1) xa[c0 + 1] = f1;
                    if (okb && v0) xb[c0] = g0;
                    if (okb && v1) xb[c0 + 1] = g1;
                    continue;
                }
                if (t < nxq + nwt) {
                    const int r = t - nxq, wi = 8 * r + fr;   // row of the right-hand side = column wi of Wp
                    const int c0 = p0 + 2 * fk;
                    if (8 * r == p0) {   // diagonal tile: I inv(L_pp)^T
                        if (wi < n) {
                            if (2 * fk >= fr && c0 < n) Wp[tri(c0, wi)] = dinv[(2 * fk) * 8 + fr];
                            if (2 * fk + 1 >= fr && c0 + 1 < n) Wp[tri(c0 + 1, wi)] = dinv[(2 * fk + 1) * 8 + fr];
                        }
                        continue;
                    }
                    const double *lrow = A + tri(min(p0 + fr, n - 1), 0) + fk;   // L(p0 + fr, q + fk): B fragment
                    double d0 = 0.0, d1 = 0.0, d2 = 0.0, d3 = 0.0;
#pragma unroll 2
                    for (int q = 8 * r; q < p0; q += 8) {   // entries left of the diagonal of Wp's transpose are structural zeros
                        const int ka = q + fk, kb = ka + 4;
                        const double xa0 = ka >= wi ? Wp[tri(ka, wi)] : 0.0, xa1 = kb >= wi ? Wp[tri(kb, wi)] : 0.0;
                        dmma884(d0, d1, xa0, lrow[q]);
                        dmma884(d2, d3, xa1, lrow[q + 4]);
                    }
                    const bool v0 = c0 < n, v1 = c0 + 1 < n;
                    const int k0 = p0 + fk, k1 = k0 + 4;
                    if (v0) Wp[tri(c0, wi)] = -(d0 + d2);   // in place, to be re-read as an A fragment
                    if (v1) Wp[tri(c0 + 1, wi)] = -(d1 + d3);
                    __syncwarp();
                    const double aa0 = k0 < n ? Wp[tri(k0, wi)] : 0.0, aa1 = k1 < n ? Wp[tri(k1, wi)] : 0.0;
                    const double bd0 = dinv[fr * 8 + fk], bd1 = dinv[fr * 8 + fk + 4];   // B[k][c] = Dinv[c][k]
                    double f0 = 0.0, f1 = 0.0;
                    dmma884(f0, f1, aa0, bd0);
                    dmma884(f0, f1, aa1, bd1);
                    __syncwarp();
                    if (v0) Wp[tri(c0, wi)] = f0;
                    if (v1) Wp[tri(c0 + 1, wi)] = f1;
                    continue;
                }
                a_tile(t - nxq - nwt + 1);
            }
        }
        CHOL_T(p0 >> 3, 4);
        __syncthreads();
        CHOL_T(p0 >> 3, 5);
    }
#ifdef SLB_CHOL_TIMING
    if (threadIdx.x == 0 && blockIdx.x == 0) ++chol_dbg_call;
#endif
}

// ---- two factorisations in lockstep -----------------------------------------------------------------------------------
// A Cholesky without right-hand sides keeps one warp busy (the diagonal-block chain) and 15 waiting.  chol(P_new) of the
// current instance and chol(P) of the NEXT instance (its record is already in shared memory) are independent, so they are
// factored panel by panel in the same phases: warp 0 owns the diagonal blocks of A1, warp 1 (another scheduler) those of
// A2, the panel solves and trailing tiles of both are spread over the other warps.  Same arithmetic per matrix as
// chol_blocked (bitwise: the per-matrix operations and their order do not depend on which warp runs them).
SLB_DEV void dual_factor_diag(double *A, int n, int p0, double a0, double a1, double *dinv, int *ok_flag, int lane) {
    const int fr = lane >> 2, fk = lane & 3;
    const int pb = min(8, n - p0);
    const int i = fr, j0 = 2 * fk, j1 = j0 + 1;
    double m0 = (i == j0) ? 1.0 : 0.0, m1 = (i == j1) ? 1.0 : 0.0;
    double di = 1.0, dj0 = 1.0, dj1 = 1.0;
    bool ok = true;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        if (k < pb) {
            const int kh = k >> 1;
            const double ak = (k & 1) ? a1 : a0;
            const double d = bcast(ak, 4 * k + kh);
            const double aik = __shfl_sync(0xffffffffu, ak, 4 * i + kh);
            ok = ok && (d > 0.0);
            if (i == k) di = d;
            if (j0 == k) dj0 = d;
            if (j1 == k) dj1 = d;
            if (k < 7) {
                const double ajk0 = __shfl_sync(0xffffffffu, ak, 4 * j0 + kh), ajk1 = __shfl_sync(0xffffffffu, ak, 4 * j1 + kh);
                const double mk0 = bcast(m0, 4 * k + fk), mk1 = bcast(m1, 4 * k + fk);
                const double v = aik * rcp_fast(d);
                if (j0 > k) a0 = fma(-v, ajk0, a0);
                if (j1 > k) a1 = fma(-v, ajk1, a1);
                const double vm = i > k ? v : 0.0;
                m0 = fma(-vm, mk0, m0);
                m1 = fma(-vm, mk1, m1);
            }
        }
    }
    double si, ri, s0, r0c, s1, r1c;
    sqrt_rsqrt(di, si, ri);
    sqrt_rsqrt(dj0, s0, r0c);
    sqrt_rsqrt(dj1, s1, r1c);
    if (i < pb) {
        if (j0 <= i) A[tri(p0 + i, p0 + j0)] = (j0 == i) ? s0 : a0 * r0c;
        if (j1 <= i) A[tri(p0 + i, p0 + j1)] = (j1 == i) ? s1 : a1 * r1c;
    }
    *reinterpret_cast<double2 *>(dinv + i * 8 + j0) = make_double2(j0 <= i ? ri * m0 : 0.0, j1 <= i ? ri * m1 : 0.0);
    ok = __all_sync(0xffffffffu, ok);
    if (!ok && lane == 0) *ok_flag = 0;
}

SLB_DEV void chol_dual(double *A1, double *A2, int n, int *ok1, int *ok2, double *PS1, double *PS2) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int fr = lane >> 2, fk = lane & 3;
    auto dinv_of = [&](double *PS, int p0) { return PS + MS_PS - 128 + 64 * ((p0 >> 3) & 1); };
    if (warp < 2) {
        double *A = warp ? A2 : A1;
        const int pb = min(8, n);
        dual_factor_diag(A, n, 0, (fr < pb && 2 * fk <= fr) ? A[tri(fr, 2 * fk)] : 0.0, (fr < pb && 2 * fk + 1 <= fr) ? A[tri(fr, 2 * fk + 1)] : 0.0,
                         dinv_of(warp ? PS2 : PS1, 0), warp ? ok2 : ok1, lane);
    }
    __syncthreads();
    for (int p0 = 0; p0 < n; p0 += 8) {
        const int pb = min(8, n - p0);
        const int r0 = p0 + pb, na = n - r0;
        const int ntl = (na + 7) >> 3;
        for (int t = warp; t < 2 * ntl; t += MS_W) {   // panel solve: rows * inv(L_pp)^T, one 8-row tile per warp
            const int m = t >= ntl, rt = t - m * ntl;
            double *A = m ? A2 : A1, *PS = m ? PS2 : PS1;
            const double *dinv = dinv_of(PS, p0);
            const int w = 8 * rt + fr, wc = min(w, na - 1);
            const double *Ai = A + tri(r0 + wc, p0);
            double x0 = 0.0, x1 = 0.0;
            dmma884(x0, x1, Ai[fk], dinv[fr * 8 + fk]);
            dmma884(x0, x1, Ai[fk + 4], dinv[fr * 8 + fk + 4]);
            __syncwarp();
            if (w < na) {
                double *Ao = A + tri(r0 + w, p0) + 2 * fk;
                Ao[0] = x0;
                Ao[1] = x1;
                *reinterpret_cast<double2 *>(PS + ps_idx(w, 2 * fk)) = make_double2(x0, x1);
            }
        }
        __syncthreads();
        const int nt = (na + 7) >> 3, ntiles = nt * (nt + 1) / 2;
        if (warp < 2) {
            if (ntiles > 0) {   // look-ahead on the next diagonal block of this warp's matrix
                double *A = warp ? A2 : A1, *PS = warp ? PS2 : PS1;
                const int rr = min(fr, na - 1), pbn = min(8, na);
                const int i = r0 + fr, j = r0 + 2 * fk;
                const bool v0 = fr < pbn && 2 * fk <= fr, v1 = fr < pbn && 2 * fk + 1 <= fr;
                const double x0 = PS[ps_idx(rr, fk)], x1 = PS[ps_idx(rr, fk + 4)];
                const double c0 = v0 ? A[tri(i, j)] : 0.0, c1 = v1 ? A[tri(i, j + 1)] : 0.0;
                double d0 = 0.0, d1 = 0.0;
                dmma884(d0, d1, x0, x0);
                dmma884(d0, d1, x1, x1);
                dual_factor_diag(A, n, r0, v0 ? c0 - d0 : 0.0, v1 ? c1 - d1 : 0.0, dinv_of(PS, r0), warp ? ok2 : ok1, lane);
            }
        } else {
            const int nat = max(ntiles - 1, 0);
            for (int t = warp - 2; t < 2 * nat; t += MS_W - 2) {
                const int m = t >= nat, tt = t - m * nat + 1;
                double *A = m ? A2 : A1, *PS = m ? PS2 : PS1;
                int tr, tc;
                tri_tile(tt, tr, tc);
                const int i0 = r0 + 8 * tr, j0 = r0 + 8 * tc;
                double d0 = 0.0, d1 = 0.0;
                const int ra = min(8 * tr + fr, na - 1), rb = min(8 * tc + fr, na - 1);
                const int i = i0 + fr, j = j0 + 2 * fk;
                const bool v0 = i < n && j <= i, v1 = i < n && j + 1 <= i;
                double *po = A + tri(min(i, n - 1), min(j, i));
                const double c0 = v0 ? po[0] : 0.0, c1 = v1 ? po[1] : 0.0;
                dmma884(d0, d1, PS[ps_idx(ra, fk)], PS[ps_idx(rb, fk)]);
                dmma884(d0, d1, PS[ps_idx(ra, fk + 4)], PS[ps_idx(rb, fk + 4)]);
                if (v0) po[0] = c0 - d0;
                if (v1) po[1] = c1 - d1;
            }
        }
        __syncthreads();
    }
}

// removeRow(2i); removeRow(2i+1) of the reference's gate loop applied to the index list kept[0..len) by one warp;
// the second index is NOT re-based (quirk Q6).  Returns the new length.
SLB_DEV int gate_remove_pair(int *kept, int len, int i, int lane) {
    for (int pass = 0; pass < 2; ++pass) {
        const int pos = 2 * i + pass, num = len - 1;
        int v[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int e = pos + lane + 32 * q;
            v[q] = e < num ? kept[e + 1] : 0;
        }
        __syncwarp();
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int e = pos + lane + 32 * q;
            if (e < num) kept[e] = v[q];
        }
        __syncwarp();
        len = num;
    }
    return len;
}

SLB_DEV int ms_qoff(int b) { return b < 4 ? (b == 0 ? 0 : b == 1 ? 3 : b == 2 ? 7 : 10) : 13 + 7 * ((b - 4) >> 1) + (((b - 4) & 1) ? 3 : 0); }
SLB_DEV bool ms_so3(int b) { return b < 4 ? b == 1 : ((b - 4) & 1); }

__global__ void __launch_bounds__(MS_T, 1) msckf_update_kernel(slb::FilterArgs a) {
    extern __shared__ __align__(16) double sm[];
    double *RA = sm, *RB = RA + MS_A, *RC = RB + MS_B, *RD = RC + MS_C;
    double *PS = RB + MS_A;   // panel staging of chol_blocked: region B is idle (or holds the compacted S' in its first MS_A slots) during every factorisation
    double *mu = RD, *zbar = mu + 84, *nu = zbar + 100, *wv = nu + 100, *dl = wv + 100, *acc = dl + 72, *ref = acc + 72,
           *invd = ref + 84;  // 104
    int *kept = reinterpret_cast<int *>(invd + 104);  // 100 ints
    int *flags = kept + 100;                          // [0] chol ok, [1] kept count, [2] outliers, [3] loop, [4] iters
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int fr = lane >> 2, fk = lane & 3;          // DMMA fragment coordinates of this lane
    const int k = a.k, N = 12 + 6 * k, QD = 13 + 7 * k, NS = 2 * N + 1, M = a.m, NF = M / 2, NB = 4 + 2 * k;
    const int NP = N * (N + 1) / 2;
    const int nrt = (N + 7) >> 3;                     // 8-row tiles of the state

    // CTA-uniform: the previous iteration already factored this instance's covariance (chol_dual, in lockstep with its own
    // chol(P_new)) and parked L at RC + MS_NXL, its pivot flag in flags[5]
    bool have_l = false;
#ifdef SLB_MSCKF_PHASES
    int ms_it = -1;
#endif
    for (int inst = blockIdx.x; inst < a.B; inst += gridDim.x) {
        double *Pg = a.P + (size_t)inst * a.pstride;
        double *mug = a.mu + (size_t)inst * a.qstride;
        const double *zg = a.z + (size_t)inst * M;
        __syncthreads();
#ifdef SLB_MSCKF_PHASES
        ++ms_it;
#endif
        MS_PH(0);
        // cp.async keeps every load of the record in flight at once
        if (have_l) {
            for (int e = tid; e < NP; e += MS_T) RA[e] = RC[MS_NXL + e];
        } else {
            for (int e = tid; e < NP; e += MS_T) cp_async8(RA + e, Pg + e);
        }
        for (int e = tid; e < QD; e += MS_T) mu[e] = mug[e];
        if (tid == 0) { flags[0] = have_l ? flags[5] : 1; flags[1] = M; flags[2] = 0; }
        cp_async_wait_all();
        __syncthreads();
        MS_PH(1);
        // ---- L = chol(Pk) (:229 -> :412), unless the previous iteration already did it ------------------
        if (!have_l) chol_blocked(RA, N, flags, invd, PS);
        have_l = false;
        int st = 0;
        if (!flags[0]) {
            if (tid == 0) a.status[inst] |= SLB_ST_CHOL_FAIL;
            continue;
        }
        MS_PH(2);
        // ---- sigma points through h (:229-232), thread per sigma point ---------------------------------
        // h = SLB_MM_MSCKF_REPROJ: feature f is landmark f seen from clone f % k (statek is not observed)
        // work item = (sigma point, clone): NS * k items over the whole CTA
        // (Skipping the (sigma point, clone) pairs the factor's column cannot reach -- 37 % of them, copies of row 0 -- was
        // tried: the uneven rounds and the extra copy pass cost more than the projections they save, 11.4k -> 15.2k cycles.)
        for (int w = tid; w < NS * k; w += MS_T) {
            const int s = w / k, c = w - s * k, j = s >= 1 ? (s - 1) >> 1 : 0;
            const double sgn = (s & 1) ? 1.0 : -1.0;
            double *Zr = RB + s * MS_ZS;
            {
                const int r0 = 12 + 6 * c;
                double d[6];
#pragma unroll
                for (int r = 0; r < 6; ++r) d[r] = (s >= 1 && r0 + r >= j) ? sgn * RA[tri(r0 + r, j)] : 0.0;
                const double *mp = mu + 13 + 7 * c;
                const double p[3] = {mp[0] + d[0], mp[1] + d[1], mp[2] + d[2]};
                double e[4], q[4];
                so3_exp(d + 3, 1.0, e);
                quat_mul(mp + 3, e, q);
                for (int f = c; f < NF; f += k) {
                    const double dv[3] = {__ldg(a.params + 3 * f) - p[0], __ldg(a.params + 3 * f + 1) - p[1],
                                          __ldg(a.params + 3 * f + 2) - p[2]};
                    double pc[3];
                    quat_rotate_inv(q, dv, pc);
                    const double iz = rcp_fast(pc[2]);
                    Zr[2 * f] = pc[0] * iz;
                    Zr[2 * f + 1] = pc[1] * iz;
                }
            }
        }
        __syncthreads();
        MS_PH(3);
        // ---- mean_z, innovation (:234-236) -------------------------------------------------------------
        if (tid < M) {
            // four interleaved partial sums: the additions of a column no longer form one 145-long dependent chain
            double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
            int t = 0;
            for (; t + 3 < NS; t += 4) {
                s0 += RB[t * MS_ZS + tid];
                s1 += RB[(t + 1) * MS_ZS + tid];
                s2 += RB[(t + 2) * MS_ZS + tid];
                s3 += RB[(t + 3) * MS_ZS + tid];
            }
            for (; t < NS; ++t) s0 += RB[t * MS_ZS + tid];
            const double s = (s0 + s1) + (s2 + s3);
            const double zb = s * (1.0 / (double)NS);
            zbar[tid] = zb;
            nu[tid] = zg[tid] - zb;
        }
        MS_PH(4);
        // ---- W_j = 0.5 (Z+_j - Z-_j) into region C ---------------------------------------------------
        //      and, in the same pass over the pair of rows, centre Z for the covariance (each element is read once; the four
        //      column chunks of a row pair are independent chains).  The pad rows NS..NSPAD-1 are zeroed so that the k-loop
        //      of S needs no bound check.
        __syncthreads();   // zbar
        for (int j = warp; j < N; j += MS_W) {
            double *zp = RB + (1 + 2 * j) * MS_ZS, *zm = zp + MS_ZS;
#pragma unroll
            for (int q = 0; q < (MS_MMAX + 31) / 32; ++q) {
                const int c = lane + 32 * q;
                if (c < M) {
                    const double vp = zp[c], vm = zm[c], zb = zbar[c];
                    RC[j * MS_ZS + c] = 0.5 * (vp - vm);
                    zp[c] = vp - zb;
                    zm[c] = vm - zb;
                }
            }
        }
        for (int e = tid; e < M; e += MS_T) RB[e] -= zbar[e];
        for (int e = tid; e < (MS_NSPAD - NS) * M; e += MS_T) RB[(NS + e / M) * MS_ZS + e % M] = 0.0;
        __syncthreads();   // W complete before the TRMM reads other warps' rows
        MS_PH(5);
        // ---- covXZ = L W (:239 -> :635-657): in-place TRMM on region C.  A warp owns an 8-column strip and
        //      walks the row tiles bottom-up (row tile tr reads only rows <= 8 tr + 7 of its own strip) ------
        for (int tc = warp; tc < ((M + 7) >> 3); tc += MS_W) {
            const int bc = min(8 * tc + fr, M - 1);   // clamped: columns >= M are never stored
            for (int tr = nrt - 1; tr >= 0; --tr) {
                const int ai = 8 * tr + fr, aic = min(ai, N - 1);
                const double *pa = RA + tri(aic, 0) + fk, *pb = RC + fk * MS_ZS + bc;
                double d0 = 0.0, d1 = 0.0;
#pragma unroll 4
                for (int k0 = 0; k0 < 8 * tr; k0 += 4) dmma884(d0, d1, pa[k0], pb[k0 * MS_ZS]);  // kk < 8 tr <= ai: inside L
#pragma unroll
                for (int k0 = 8 * tr; k0 < 8 * tr + 8; k0 += 4) {                                 // the diagonal tile
                    const int kk = k0 + fk;
                    const double av = kk <= aic ? pa[k0] : 0.0;
                    const double bv = kk < N ? pb[k0 * MS_ZS] : 0.0;
                    dmma884(d0, d1, av, bv);
                }
                __syncwarp();
                const int oc = 8 * tc + 2 * fk;
                if (ai < N) {
                    if (oc < M) RC[ai * MS_ZS + oc] = d0;
                    if (oc + 1 < M) RC[ai * MS_ZS + oc + 1] = d1;
                }
                __syncwarp();
            }
        }
        __syncthreads();
        MS_PH(6);
        // ---- S = 0.5 Zc^T Zc + R (:238) into region A (L is dead): lower 8x8 tiles, K = sigma points ----------
        {
            const int nt = (M + 7) >> 3, ntiles = nt * (nt + 1) / 2;
            for (int t = warp; t < ntiles; t += MS_W) {
                int tr, tc;
                tri_tile(t, tr, tc);
                // rows / columns beyond M only feed outputs that are dropped below (D(i,j) uses row i of A and column j
                // of B only), so their addresses are merely clamped into the buffer: the loop is 2 LDS + 1 DMMA
                const double *pa = RB + fk * MS_ZS + min(8 * tr + fr, M - 1), *pb = RB + fk * MS_ZS + min(8 * tc + fr, M - 1);
                double d0 = 0.0, d1 = 0.0;
#pragma unroll 4
                for (int k0 = 0; k0 < MS_NSPAD; k0 += 4) dmma884(d0, d1, pa[k0 * MS_ZS], pb[k0 * MS_ZS]);
                const int r = 8 * tr + fr, c = 8 * tc + 2 * fk;
                if (r < M) {
                    if (c <= r) RA[tri(r, c)] = 0.5 * d0 + __ldg(a.R + r * M + c);
                    if (c + 1 <= r) RA[tri(r, c + 1)] = 0.5 * d1 + __ldg(a.R + r * M + c + 1);
                }
            }
        }
        __syncthreads();
        MS_PH(7);
        // ---- removeOutliers (:241 -> :723-754), index quirk Q6 reproduced ---------------------------------
        if (a.gate) {
            // every feature against the 2-dof 5% bound in parallel first: while nothing is rejected the reference's
            // sequential scan keeps the identity indexing, so "all accepted" needs no scan at all
            bool rej = false;
            if (tid < NF) {
                const int ia = 2 * tid, ib = ia + 1;
                const double s00 = RA[tri(ia, ia)], s11 = RA[tri(ib, ib)], s10 = RA[tri(ib, ia)];
                const double det = s00 * s11 - s10 * s10;
                const double v0 = nu[ia], v1 = nu[ib];
                const double m2 = (v0 * (s11 * v0 - s10 * v1) + v1 * (s00 * v1 - s10 * v0)) / det;
                rej = !(m2 < 5.99);
            }
            if (__syncthreads_or(rej) && warp == 0) {
                // the reference's sequential scan, 32 positions at a time: every lane tests one position against the
                // current index list, the first rejection (if any) is applied, and the scan resumes from there
                int len = M, out = 0, i = 0;
                for (int e = lane; e < M; e += 32) kept[e] = e;
                __syncwarp();
                while (i < len / 2) {
                    const int ii = i + lane;
                    bool rj = false;
                    if (ii < len / 2) {
                        const int ia = kept[2 * ii], ib = kept[2 * ii + 1];
                        const double s00 = RA[tri(ia, ia)], s11 = RA[tri(ib, ib)], s10 = ib > ia ? RA[tri(ib, ia)] : RA[tri(ia, ib)];
                        const double det = s00 * s11 - s10 * s10;
                        const double v0 = nu[ia], v1 = nu[ib];
                        const double m2 = (v0 * (s11 * v0 - s10 * v1) + v1 * (s00 * v1 - s10 * v0)) / det;
                        rj = !(m2 < 5.99);
                    }
                    const unsigned bal = __ballot_sync(0xffffffffu, rj);
                    if (!bal) {
                        i += 32;
                        continue;
                    }
                    i += __ffs(bal) - 1;
                    len = gate_remove_pair(kept, len, i, lane);
                    ++out;
                }
                if (lane == 0) { flags[1] = len; flags[2] = out; }
            }
        }
        __syncthreads();
        MS_PH(8);
        const int mk = flags[1];
        if (tid == 0) a.outliers[inst] = flags[2];
        if (mk <= 0) continue;  // :250 nothing left to update with
        double *Sp = RA, *Xz = RC;  // S' (packed, stride implicit) and covXZ' (row stride MS_ZS)
        if (mk < M) {
            // compact S -> region B (Z is dead), covXZ in place (kept[] is increasing, kept[p] >= p)
            for (int e = tid; e < mk * (mk + 1) / 2; e += MS_T) {
                int r = (int)((sqrtf(8.0f * e + 1.0f) - 1.0f) * 0.5f);
                r += (tri(r + 1, 0) <= e) - (tri(r, 0) > e);
                const int c = e - tri(r, 0);
                RB[e] = RA[tri(kept[r], kept[c])];
            }
            // a warp per row of covXZ: the row is gathered into registers before it is overwritten (m <= 128 = 4 per lane)
            for (int i = warp; i < N; i += MS_W) {
                double *row = RC + i * MS_ZS;
                double v[4];
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const int pp = lane + 32 * q;
                    v[q] = pp < mk ? row[kept[pp]] : 0.0;
                }
                __syncwarp();
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const int pp = lane + 32 * q;
                    if (pp < mk) row[pp] = v[q];
                }
            }
            if (tid < mk) wv[tid] = nu[kept[tid]];
            __syncthreads();
            if (tid < mk) nu[tid] = wv[tid];
            Sp = RB;
            __syncthreads();
        }
        // ---- Ls = chol(S') and Y = covXZ' Ls^-T in one sweep: the rows of covXZ' are carried through the panel solves and
        //      trailing updates of the factorisation.  The innovation rides along as one more row (kept in wv: region C has
        //      exactly N rows): [covXZ; nu^T] Ls^-T has w^T = (Ls^-1 nu)^T as its last row.
        if (tid < mk) wv[tid] = nu[tid];
        __syncthreads();
        MS_PH(9);
        chol_blocked(Sp, mk, flags, invd, PS, Xz, N, MS_ZS, wv);
        if (!flags[0]) {
            if (tid == 0) a.status[inst] |= SLB_ST_CHOL_FAIL;
            continue;
        }
        MS_PH(10);
        // region B (the compacted S' and the panel staging) is dead: the next instance's covariance record goes there now, to be
        // factored together with this instance's P_new below
        const bool more = inst + (int)gridDim.x < a.B;
        if (more) {
            const double *Pn = a.P + (size_t)(inst + gridDim.x) * a.pstride;
            for (int e = tid; e < NP; e += MS_T) cp_async8(RB + e, Pn + e);
            if (tid == 0) flags[5] = 1;
        }
        // ---- delta = Y w, w = the extra row of the solve ---------------------------------------------------------
        for (int i = warp; i < N; i += MS_W) {
            double s = 0.0;
            for (int q = lane; q < mk; q += 32) s += Xz[i * MS_ZS + q] * wv[q];
            s = warp_sum(s);
            if (lane == 0) dl[i] = s;
        }
        MS_PH(11);
        // ---- P_new = Pk - Y Y^T (:262) into region A from the HBM record: lower 8x8 tiles, K = mk ------------
        __syncthreads();
        {
            const int ntiles = nrt * (nrt + 1) / 2;
            for (int t = warp; t < ntiles; t += MS_W) {
                int tr, tc;
                tri_tile(t, tr, tc);
                const int ai = 8 * tr + fr;
                const double *pa = Xz + min(ai, N - 1) * MS_ZS + fk, *pb = Xz + min(8 * tc + fr, N - 1) * MS_ZS + fk;
                double d0 = 0.0, d1 = 0.0;
                const int r = ai, c = 8 * tc + 2 * fk;
                // the record's entries are requested before the k-loop so that their L2 latency hides behind it
                const double g0 = (r < N && c <= r) ? Pg[tri(r, c)] : 0.0, g1 = (r < N && c + 1 <= r) ? Pg[tri(r, c + 1)] : 0.0;
                const int kfull = mk & ~3;   // mk is even: at most one ragged k-step
#pragma unroll 4
                for (int k0 = 0; k0 < kfull; k0 += 4) dmma884(d0, d1, pa[k0], pb[k0]);
                if (kfull < mk) {
                    const bool in = kfull + fk < mk;
                    dmma884(d0, d1, in ? pa[kfull] : 0.0, in ? pb[kfull] : 0.0);
                }
                if (r < N) {
                    if (c <= r) RA[tri(r, c)] = g0 - d0;
                    if (c + 1 <= r) RA[tri(r, c + 1)] = g1 - d1;
                }
            }
        }
        cp_async_wait_all();
        __syncthreads();
        MS_PH(12);
        // ---- applyDelta(K nu) (:263 -> :659-666): L2 = chol(P_new), X = mu [+] (delta +- L2 e_j).  A factorisation without
        //      right-hand sides keeps one warp busy and fifteen waiting, so chol(P) of the NEXT instance runs in lockstep with
        //      it (chol_dual) and is parked in region C (Y is dead; the mean's partial sums stay below MS_NXL) ----------------
        if (more) {
            chol_dual(RA, RB, N, flags, flags + 5, PS, PS + MS_PS);
            for (int e = tid; e < NP; e += MS_T) RC[MS_NXL + e] = RB[e];
            have_l = true;
            __syncthreads();   // region B is about to receive the sigma points
        } else {
            chol_blocked(RA, N, flags, invd, PS);
        }
        if (!flags[0]) {
            if (tid == 0) a.status[inst] |= SLB_ST_CHOL_FAIL;
            continue;
        }
        MS_PH(13);
        for (int w = tid; w < NS * NB; w += MS_T) {   // work item = (block, sigma point), block-major: a warp's 32 items share
                                                      // the block type (SO3 / vector) instead of diverging over both paths
            const int b = w / NS, s = w - b * NS, j = s >= 1 ? (s - 1) >> 1 : 0;
            const double sgn = (s & 1) ? 1.0 : -1.0;
            double *X = RB + s;   // Xt[scalar][s]
            {
                double d[3];
#pragma unroll
                for (int r = 0; r < 3; ++r) d[r] = dl[3 * b + r] + ((s >= 1 && 3 * b + r >= j) ? sgn * RA[tri(3 * b + r, j)] : 0.0);
                const int qo = ms_qoff(b);
                if (ms_so3(b)) {
                    double e[4], q[4];
                    so3_exp(d, 1.0, e);
                    quat_mul(mu + qo, e, q);
                    X[qo * MS_XS] = q[0]; X[(qo + 1) * MS_XS] = q[1]; X[(qo + 2) * MS_XS] = q[2]; X[(qo + 3) * MS_XS] = q[3];
                } else {
                    X[qo * MS_XS] = mu[qo] + d[0]; X[(qo + 1) * MS_XS] = mu[qo + 1] + d[1]; X[(qo + 2) * MS_XS] = mu[qo + 2] + d[2];
                }
            }
        }
        __syncthreads();
        MS_PH(14);
        // manifold mean (:499-525): ref = X0; do { d = mean(Xi [-] ref); ref [+]= d } while (|d| > 1e-6 ...)
        for (int e = tid; e < QD; e += MS_T) ref[e] = RB[e * MS_XS];
        __syncthreads();
        // Work item = (block b, group g): group g sums X_s [-] ref over the sigma points s = g, g + G, ... in that order and
        // parks its partial in region C (Y is dead); the partials are then added in group order, so the result of an
        // instance does not depend on scheduling (bitwise reproducible across batch sizes and GPUs).
        double *part = RC;
        const int G = min(MS_T / NB, 32);
        const int mb = tid / G, mg = tid - mb * G;
        int iters = 0;
        while (true) {
            if (mb < NB) {
                const int qo = ms_qoff(mb);
                double s0 = 0.0, s1 = 0.0, s2 = 0.0;
                if (ms_so3(mb)) {
                    for (int sp = mg; sp < NS; sp += G) {
                        const double *X = RB + qo * MS_XS + sp;
                        const double xq[4] = {X[0], X[MS_XS], X[2 * MS_XS], X[3 * MS_XS]};
                        double r[4], d[3];
                        quat_cmul(ref + qo, xq, r);
                        so3_log(r, d);
                        s0 += d[0]; s1 += d[1]; s2 += d[2];
                    }
                } else {
                    for (int sp = mg; sp < NS; sp += G) {
                        const double *X = RB + qo * MS_XS + sp;
                        s0 += X[0] - ref[qo]; s1 += X[MS_XS] - ref[qo + 1]; s2 += X[2 * MS_XS] - ref[qo + 2];
                    }
                }
                double *pp = part + mg * MS_NMAX + 3 * mb;
                pp[0] = s0; pp[1] = s1; pp[2] = s2;
            }
            __syncthreads();
            if (tid < NB) {
                const int b = tid, qo = ms_qoff(b);
                const double wn = 1.0 / (double)NS;
                double d[3] = {0.0, 0.0, 0.0};
                for (int g = 0; g < G; ++g) {
                    const double *pp = part + g * MS_NMAX + 3 * b;
                    d[0] += pp[0]; d[1] += pp[1]; d[2] += pp[2];
                }
                d[0] *= wn; d[1] *= wn; d[2] *= wn;
                dl[3 * b] = d[0]; dl[3 * b + 1] = d[1]; dl[3 * b + 2] = d[2];
                if (ms_so3(b)) {
                    double e[4], q[4];
                    so3_exp(d, 1.0, e);
                    quat_mul(ref + qo, e, q);
                    ref[qo] = q[0]; ref[qo + 1] = q[1]; ref[qo + 2] = q[2]; ref[qo + 3] = q[3];
                } else {
                    ref[qo] += d[0]; ref[qo + 1] += d[1]; ref[qo + 2] += d[2];
                }
            }
            __syncthreads();
            // |d|: every warp computes it for itself (same operations, same result), so the loop needs no third barrier
            double n2 = 0.0;
            for (int e = lane; e < N; e += 32) n2 = fma(dl[e], dl[e], n2);
#pragma unroll
            for (int o = 16; o; o >>= 1) n2 += __shfl_xor_sync(0xffffffffu, n2, o);
            if (!(sqrt(n2) > 1e-6 && ++iters < 10000)) break;
        }
        MS_PH(15);
        if (iters >= 10000) st |= SLB_ST_MEAN_NOCONV;
        // deviations d_s = X_s [-] mean, in place (72 <= 83 slots per sigma point); the pad rows NS..NSPAD-1 are zeroed.
        // Thread (g, sp), g = tid / NSPAD < 3, takes the blocks b = g, g + 3, ... of sigma point sp (a warp's lanes walk the same
        // block sequence: no divergence between the SO3 and the vector path, no index divisions).  Every block is evaluated
        // into registers first and written after a barrier: the tangent slots 3b..3b+2 overlap q-blocks other threads read.
        {
            constexpr int DEV_G = MS_T / MS_NSPAD, DEV_R = (4 + 2 * 10 + DEV_G - 1) / DEV_G;   // 3 groups, <= 8 blocks each
            const int g = tid / MS_NSPAD, sp = tid - g * MS_NSPAD;
            const bool on = g < DEV_G && sp < NS;
            double dv[DEV_R][3];
#pragma unroll
            for (int t = 0; t < DEV_R; ++t) {
                const int b = g + DEV_G * t;
                dv[t][0] = dv[t][1] = dv[t][2] = 0.0;
                if (on && b < NB) {
                    const int qo = ms_qoff(b);
                    const double *X = RB + qo * MS_XS + sp;
                    if (ms_so3(b)) {
                        const double xq[4] = {X[0], X[MS_XS], X[2 * MS_XS], X[3 * MS_XS]};
                        double r[4];
                        quat_cmul(ref + qo, xq, r);
                        so3_log(r, dv[t]);
                    } else {
                        dv[t][0] = X[0] - ref[qo]; dv[t][1] = X[MS_XS] - ref[qo + 1]; dv[t][2] = X[2 * MS_XS] - ref[qo + 2];
                    }
                }
            }
            __syncthreads();
#pragma unroll
            for (int t = 0; t < DEV_R; ++t) {
                const int b = g + DEV_G * t;
                if (on && b < NB) {
                    double *X = RB + 3 * b * MS_XS + sp;   // Dt[tangent scalar][sp]
                    X[0] = dv[t][0]; X[MS_XS] = dv[t][1]; X[2 * MS_XS] = dv[t][2];
                }
            }
            for (int e = tid; e < (MS_NSPAD - NS) * N; e += MS_T) RB[(e / (MS_NSPAD - NS)) * MS_XS + NS + e % (MS_NSPAD - NS)] = 0.0;
        }
        __syncthreads();
        MS_PH(16);
        // ---- Pk = 0.5 sum d d^T (:574-589) straight to the HBM record: lower 8x8 tiles, K = sigma points ------
        {
            const int ntiles = nrt * (nrt + 1) / 2;
            for (int t = warp; t < ntiles; t += MS_W) {
                int tr, tc;
                tri_tile(t, tr, tc);
                const int ar = 8 * tr + fr;
                const double *pa = RB + min(ar, N - 1) * MS_XS + fk, *pb = RB + min(8 * tc + fr, N - 1) * MS_XS + fk;
                double d0 = 0.0, d1 = 0.0;
#pragma unroll 4
                for (int k0 = 0; k0 < MS_NSPAD; k0 += 4) dmma884(d0, d1, pa[k0], pb[k0]);  // pad sigma points are zero
                const int r = ar, c = 8 * tc + 2 * fk;
                if (r < N) {
                    if (c <= r) Pg[tri(r, c)] = 0.5 * d0;
                    if (c + 1 <= r) Pg[tri(r, c + 1)] = 0.5 * d1;
                }
            }
        }
        MS_PH(17);
        bool finite = true;
        for (int e = tid; e < QD; e += MS_T) {
            mug[e] = ref[e];
            finite = finite && isfinite(ref[e]);
        }
        if (!finite) st |= SLB_ST_NONFINITE;
        if (st) atomicOr(a.status + inst, st);
        MS_PH(18);
    }
}


// =====================================================================================================
// SURVEY 8(f) row f1: Msckf::update, EKF flavour (Msckf.hpp:297-349) -- h(mu, H) with its Jacobian, removeOutliers on
// H (:756-792: information = (H P H^T + R)^-1 computed once and never compacted, row-index quirk Q6), reduceDimension
// (:794-816: Householder QR of H, thin Q, H <- R(0:N,0:N), nu <- Q^T nu, R <- Q^T R Q), S = H P H^T + R,
// K = P H^T S^-1, Pk -= K S K^T, mu = mu [+] K nu.  One instance per CTA, everything in shared memory:
//   RA  2632 : Pk (packed lower), read-only
//   RS  5056 : S100 -> L100 (information) ... later Rr -> S72 -> Ls
//   RH  7600 : H (100 x 76) ... later thin Q ... later covXZ = P Hr^T -> Y = covXZ Ls^-T
//   RQ  7600 : T = H P ... L100^-1 (packed) ... compacted H -> R1 (Householder QR in place)
// Same algebra shortcuts as the UKF flavour (quirk Q9): the 2x2 diagonal blocks of the information matrix come from
// the triangular inverse of chol(S100) (information_ff = W_f^T W_f), and with S = Ls Ls^T, Y = (P Hr^T) Ls^-T the
// gain algebra is Pk -= Y Y^T, delta = Y (Ls^-1 nu).  The measurement model is SLB_MM_MSCKF_REPROJ with its analytic
// Jacobian (d pc = -R^T dp + [pc]x dtheta); H has one 2 x 6 block per feature, which the H P H^T products exploit.
// =====================================================================================================
constexpr int ME_QP = MS_T / 80;  // threads sharing a column in the Householder phases (rows i = first + part mod QP)
constexpr int ME_HS = 76;  // row stride of H / Q / covXZ (= 12 mod 16: conflict-free DMMA fragment loads)
constexpr int ME_RA = 2632, ME_RS = 5056, ME_RH = MS_MMAX * ME_HS, ME_RQ = MS_MMAX * ME_HS, ME_RD = 2304;
constexpr int ME_SMEM_DOUBLES = ME_RA + ME_RS + ME_RH + ME_RQ + ME_RD + MS_PS;
static_assert(ME_SMEM_DOUBLES * 8 <= 227 * 1024, "MSCKF EKF update working set exceeds shared memory");

// flag[0] = 1 when the shared m x m measurement noise matrix is diagonal, flag[1] = 1 when it is sigma^2 I
__global__ void msckf_rdiag_kernel(const double *R, int m, int32_t *flag) {
    __shared__ int off, uneq;
    if (threadIdx.x == 0) { off = 0; uneq = 0; }
    __syncthreads();
    const double r0 = R[0];
    int mine = 0, ne = 0;
    for (int e = threadIdx.x; e < m * m; e += blockDim.x) {
        if (e / m != e % m) { if (R[e] != 0.0) mine = 1; }
        else if (R[e] != r0) ne = 1;
    }
    if (mine) off = 1;
    if (ne) uneq = 1;
    __syncthreads();
    if (threadIdx.x == 0) { flag[0] = off ? 0 : 1; flag[1] = (off || uneq || !(r0 > 0.0)) ? 0 : 1; }
}

__global__ void __launch_bounds__(MS_T, 1) msckf_ekf_update_kernel(slb::FilterArgs a) {
    extern __shared__ __align__(16) double sm[];
    double *RA = sm, *RS = RA + ME_RA, *RH = RS + ME_RS, *RQ = RH + ME_RH, *RD = RQ + ME_RQ, *PS = RD + ME_RD;
    double *mu = RD, *nu = mu + 84, *wv = nu + 100, *dl = wv + 100, *invd = dl + 72, *tau = invd + 104, *Hb = tau + 72,
           *info = Hb + 600, *T3 = info + 152, *scal = T3 + 800;  // scal: 8
    int *kept = reinterpret_cast<int *>(scal + 8);  // 100 ints
    int *flags = kept + 100;                        // [0] chol ok, [1] kept count, [2] outliers
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int fr = lane >> 2, fk = lane & 3;
    const int k = a.k, N = 12 + 6 * k, QD = 13 + 7 * k, M = a.m, NF = M / 2, NB = 4 + 2 * k;
    const int NP = N * (N + 1) / 2;
    const int nrt = (N + 7) >> 3;
    auto Psym = [&](int i, int j) { return i >= j ? RA[tri(i, j)] : RA[tri(j, i)]; };
    constexpr int QP = ME_QP;

    // With R = sigma^2 I (flagged once per launch by msckf_rdiag_kernel) the update takes the direct form (see below)
    const bool direct = a.misc[1] != 0;
    bool fetched = false;   // CTA-uniform: RQ holds (or is receiving) this instance's covariance record, see below
    for (int inst = blockIdx.x; inst < a.B; inst += gridDim.x) {
        double *Pg = a.P + (size_t)inst * a.pstride;
        double *mug = a.mu + (size_t)inst * a.qstride;
        const double *zg = a.z + (size_t)inst * M;
        __syncthreads();
        if (fetched) {
            cp_async_wait_all();
            __syncthreads();
            for (int e = tid; e < NP; e += MS_T) RA[e] = RQ[e];
        } else {
            for (int e = tid; e < NP; e += MS_T) RA[e] = Pg[e];
        }
        fetched = false;
        for (int e = tid; e < QD; e += MS_T) mu[e] = mug[e];
        if (!direct)   // the dense H is only read by the QR path
            for (int e = tid; e < M * ME_HS; e += MS_T) RH[e] = 0.0;
        if (tid == 0) { flags[0] = 1; flags[1] = M; flags[2] = 0; }
        __syncthreads();
        // ---- mean_z = h(mu, H), innovation (:311-313): thread per feature ---------------------------------------
        if (tid < NF) {
            const int f = tid, c = f % k;
            const double *mp = mu + 13 + 7 * c, *q = mp + 3;
            const double dv[3] = {__ldg(a.params + 3 * f) - mp[0], __ldg(a.params + 3 * f + 1) - mp[1],
                                  __ldg(a.params + 3 * f + 2) - mp[2]};
            double pc[3];
            quat_rotate_inv(q, dv, pc);
            const double iz = 1.0 / pc[2];
            const double z0 = pc[0] * iz, z1 = pc[1] * iz;
            nu[2 * f] = zg[2 * f] - z0;
            nu[2 * f + 1] = zg[2 * f + 1] - z1;
            // d pc / d(dp) = -R^T, d pc / d(dtheta) = [pc]x
            const double w = q[0], x = q[1], y = q[2], zq = q[3];
            const double tx = 2 * x, ty = 2 * y, tz = 2 * zq;
            const double twx = tx * w, twy = ty * w, twz = tz * w, txx = tx * x, txy = ty * x, txz = tz * x, tyy = ty * y,
                         tyz = tz * y, tzz = tz * zq;
            const double Rm[9] = {1 - (tyy + tzz), txy - twz, txz + twy, txy + twz, 1 - (txx + tzz), tyz - twx,
                                  txz - twy,       tyz + twx, 1 - (txx + tyy)};
            double J[3][6];
#pragma unroll
            for (int r = 0; r < 3; ++r)
#pragma unroll
                for (int cc = 0; cc < 3; ++cc) J[r][cc] = -Rm[cc * 3 + r];
            J[0][3] = 0.0; J[0][4] = -pc[2]; J[0][5] = pc[1];
            J[1][3] = pc[2]; J[1][4] = 0.0; J[1][5] = -pc[0];
            J[2][3] = -pc[1]; J[2][4] = pc[0]; J[2][5] = 0.0;
#pragma unroll
            for (int cc = 0; cc < 6; ++cc) {
                const double h0 = iz * (J[0][cc] - z0 * J[2][cc]), h1 = iz * (J[1][cc] - z1 * J[2][cc]);
                Hb[(2 * f) * 6 + cc] = h0;
                Hb[(2 * f + 1) * 6 + cc] = h1;
                if (!direct) {
                    RH[(2 * f) * ME_HS + 12 + 6 * c + cc] = h0;
                    RH[(2 * f + 1) * ME_HS + 12 + 6 * c + cc] = h1;
                }
            }
        }
        __syncthreads();
        int mk = M;
        // in the direct form the dense H in RH is not needed, so the gate's L^-1 goes there and T = H P survives in RQ to be
        // reused as (P Hc^T)^T
        double *Wq = direct ? RH : RQ;
        if (a.gate) {
            // ---- information = (H P H^T + R)^-1 (:765-766).  T = H P over the clone columns (6 FMA per entry) ------
            // the two rows of a feature share their six rows of P: one item = (feature, column)
            for (int e = tid; e < NF * (N - 12); e += MS_T) {
                const int f = e / (N - 12), j = 12 + (e - f * (N - 12));
                const int a0 = 12 + 6 * (f % k);
                double s0 = 0.0, s1 = 0.0;
#pragma unroll
                for (int u = 0; u < 6; ++u) {
                    const double pv = Psym(a0 + u, j);
                    s0 = fma(Hb[(2 * f) * 6 + u], pv, s0);
                    s1 = fma(Hb[(2 * f + 1) * 6 + u], pv, s1);
                }
                RQ[(2 * f) * ME_HS + j] = s0;
                RQ[(2 * f + 1) * ME_HS + j] = s1;
            }
            __syncthreads();
            for (int e = tid; e < M * (M + 1) / 2; e += MS_T) {
                int r = (int)((sqrtf(8.0f * e + 1.0f) - 1.0f) * 0.5f);
                r += (tri(r + 1, 0) <= e) - (tri(r, 0) > e);
                const int c = e - tri(r, 0);
                const int a1 = 12 + 6 * ((c >> 1) % k);
                double sacc = __ldg(a.R + r * M + c);
#pragma unroll
                for (int v = 0; v < 6; ++v) sacc = fma(RQ[r * ME_HS + a1 + v], Hb[c * 6 + v], sacc);
                RS[e] = sacc;
            }
            __syncthreads();
            // W = L^-1 (packed lower in RQ; T is consumed) comes out of the same sweep: the identity is carried through the
            // factorisation as a right-hand side (chol_blocked), so the inverse costs no serial chain of its own
            chol_blocked(RS, M, flags, invd, PS, nullptr, 0, 0, nullptr, Wq);
            if (!flags[0]) {
                if (tid == 0) a.status[inst] |= SLB_ST_CHOL_FAIL;
                continue;
            }
            // 2x2 diagonal blocks of the information matrix: info_f = W[:, 2f:2f+2]^T W[:, 2f:2f+2]
            bool rej = false;
            if (tid < ((8 * NF + 31) & ~31)) {   // 8 threads per feature split the rows; whole warps take the branch
                const int f = tid >> 3, part = tid & 7, ia = 2 * f, ib = ia + 1;
                double i00 = 0.0, i10 = 0.0, i11 = 0.0;
                if (part == 0 && f < NF) {
                    const double wa = Wq[tri(ia, ia)];
                    i00 = wa * wa;
                }
                for (int r = ib + part; r < (f < NF ? M : 0); r += 8) {
                    const double wa = Wq[tri(r, ia)], wb = Wq[tri(r, ib)];
                    i00 = fma(wa, wa, i00);
                    i10 = fma(wa, wb, i10);
                    i11 = fma(wb, wb, i11);
                }
#pragma unroll
                for (int o = 4; o; o >>= 1) {
                    i00 += __shfl_xor_sync(0xffffffffu, i00, o);
                    i10 += __shfl_xor_sync(0xffffffffu, i10, o);
                    i11 += __shfl_xor_sync(0xffffffffu, i11, o);
                }
                if (part == 0 && f < NF) {
                    info[3 * f] = i00; info[3 * f + 1] = i10; info[3 * f + 2] = i11;
                    const double v0 = nu[ia], v1 = nu[ib];
                    const double m2 = v0 * (i00 * v0 + i10 * v1) + v1 * (i10 * v0 + i11 * v1);
                    rej = !(m2 < 5.99);
                }
            }
            // while nothing is rejected the sequential scan keeps the identity indexing: "all accepted" needs no scan
            if (__syncthreads_or(rej) && warp == 0) {
                int len = M, out = 0, i = 0;
                for (int e = lane; e < M; e += 32) kept[e] = e;
                __syncwarp();
                while (i < len / 2) {  // 32 scan positions per round, the first rejection is applied (see the UKF flavour)
                    const int ii = i + lane;
                    bool rj = false;
                    if (ii < len / 2) {
                        const double v0 = nu[kept[2 * ii]], v1 = nu[kept[2 * ii + 1]];
                        const double i00 = info[3 * ii], i10 = info[3 * ii + 1], i11 = info[3 * ii + 2];  // position, not feature (:773)
                        const double m2 = v0 * (i00 * v0 + i10 * v1) + v1 * (i10 * v0 + i11 * v1);
                        rj = !(m2 < 5.99);
                    }
                    const unsigned bal = __ballot_sync(0xffffffffu, rj);
                    if (!bal) {
                        i += 32;
                        continue;
                    }
                    i += __ffs(bal) - 1;
                    len = gate_remove_pair(kept, len, i, lane);  // removeRow(2i); removeRow(2i+1): not re-based (Q6)
                    ++out;
                }
                if (lane == 0) { flags[1] = len; flags[2] = out; }
            }
            __syncthreads();
            mk = flags[1];
        }
        if (tid == 0) a.outliers[inst] = flags[2];
        if (mk <= 0) continue;  // :322 nothing left
        if (mk < N) {           // :808 R.block(0,0,N,N) needs rows >= DOF
            if (tid == 0) a.status[inst] |= SLB_ST_QR_ROWS;
            continue;
        }
        const bool compact = mk < M;
        // With R = sigma^2 I (flagged once per launch) the QR compression is lossless: the rows it discards are orthogonal to
        // range(H) and uncorrelated with the ones it keeps, so the update equals the plain Kalman update on the (compacted) rows,
        //   S' = Hc P Hc^T + R',  K = P Hc^T S'^-1,
        // to rounding (3e-15 against the QR form on the config-3 scenario).  That needs no Householder QR, no thin Q, no
        // Q^T R Q and no second factorisation when nothing was rejected: the Cholesky factor of S from the outlier gate is reused.
        double *Yb = RH;   // Y = covXZ Ls^-T: base, row stride, number of measurement rows it was solved against
        int ys = ME_HS, mq = N;
        bool solved = false;   // the triangular solve was folded into the factorisation (chol_blocked with right-hand sides)
        if (direct) {
            // covXZ' = P Hc^T (N x mk), 6 FMA per entry.  After the gate its clone rows are the (compacted) transpose of T, which
            // still sits in RQ: they are copied into RH (the triangular inverse that lived there is consumed) and only the 12
            // statek rows are computed; without the gate everything is computed, into RQ.
            Yb = a.gate ? RH : RQ; ys = MS_ZS; mq = mk;
            const int ncomp = a.gate ? 12 : N;   // rows computed from scratch
            for (int e = tid; e < ncomp * mk; e += MS_T) {
                const int i = e / mk, pcol = e - i * mk, r = compact ? kept[pcol] : pcol;
                const int a0 = 12 + 6 * ((r >> 1) % k);
                double sacc = 0.0;
#pragma unroll
                for (int u = 0; u < 6; ++u) sacc = fma(Hb[r * 6 + u], Psym(a0 + u, i), sacc);
                Yb[i * MS_ZS + pcol] = sacc;
            }
            if (a.gate) {
                for (int e = tid; e < (N - 12) * mk; e += MS_T) {
                    const int pcol = e / (N - 12), i = 12 + (e - pcol * (N - 12));   // consecutive threads read consecutive T entries
                    Yb[i * MS_ZS + pcol] = RQ[(compact ? kept[pcol] : pcol) * ME_HS + i];
                }
            }
            if (tid < mk) wv[tid] = nu[compact ? kept[tid] : tid];
            __syncthreads();
            if (tid < mk) {
                nu[tid] = wv[tid];
                Yb[N * ys + tid] = wv[tid];   // the innovation rides along as row N of the solve (see below)
            }
            if (a.gate && inst + (int)gridDim.x < a.B) {
                // T is consumed: RQ is idle for the rest of this instance and receives the next instance's covariance record
                const double *Pn = a.P + (size_t)(inst + gridDim.x) * a.pstride;
                for (int e = tid; e < NP; e += MS_T) cp_async8(RQ + e, Pn + e);
                fetched = true;
            }
            if (compact || !a.gate) {
                // S' = Hc covXZ' + R' (packed lower) and its Cholesky factor; otherwise RS still holds chol(S) from the gate
                for (int e = tid; e < mk * (mk + 1) / 2; e += MS_T) {
                    int pr = (int)((sqrtf(8.0f * e + 1.0f) - 1.0f) * 0.5f);
                    pr += (tri(pr + 1, 0) <= e) - (tri(pr, 0) > e);
                    const int pc = e - tri(pr, 0);
                    const int rr = compact ? kept[pr] : pr, rc = compact ? kept[pc] : pc;
                    const int a0 = 12 + 6 * ((rr >> 1) % k);
                    double sacc = __ldg(a.R + (size_t)rr * M + rc);
#pragma unroll
                    for (int u = 0; u < 6; ++u) sacc = fma(Hb[rr * 6 + u], Yb[(a0 + u) * MS_ZS + pc], sacc);
                    RS[e] = sacc;
                }
                __syncthreads();
                chol_blocked(RS, mk, flags, invd, PS, Yb, N, ys, Yb + N * ys);
                solved = true;
                if (!flags[0]) {
                    if (tid == 0) a.status[inst] |= SLB_ST_CHOL_FAIL;
                    continue;
                }
            } else {
                __syncthreads();
            }
        } else {
        // ---- compacted H -> RQ, compacted innovation -------------------------------------------------------------
        for (int e = tid; e < mk * N; e += MS_T) {
            const int r = e / N, c = e - r * N;
            RQ[r * ME_HS + c] = RH[(compact ? kept[r] : r) * ME_HS + c];
        }
        // the innovation rides along as column N of RQ (the row stride leaves room): Q^T is applied to it with the same
        // code as to the matrix columns
        if (tid < mk) RQ[tid * ME_HS + N] = nu[compact ? kept[tid] : tid];
        __syncthreads();
        // ---- reduceDimension (:794-816): Householder QR of RQ (mk x N) in place.  Per column: partial dot products
        //      (QP threads per column), sync, rank-1 update + the partial norms of the next column, sync, rescale of
        //      the finished column + the next reflector's scalars, sync ----------------------------------------------------
        auto reflector = [&](double c0, double t, double *out, int kcol) {  // Eigen makeHouseholderInPlace
            if (t <= 2.2250738585072014e-308) {
                out[0] = 0.0;  // tau
                out[1] = 0.0;  // 1 / (c0 - beta)
                out[2] = c0;   // beta
            } else {
                double beta = sqrt(fma(c0, c0, t));
                if (c0 >= 0.0) beta = -beta;
                out[0] = (beta - c0) / beta;
                out[1] = 1.0 / (c0 - beta);
                out[2] = beta;
            }
            tau[kcol] = out[0];
        };
        if (warp == 0) {
            double t = 0.0;
            for (int i = 1 + lane; i < mk; i += 32) {
                const double v = RQ[i * ME_HS];
                t = fma(v, v, t);
            }
            t = warp_sum(t);
            if (lane == 0) reflector(RQ[0], t, scal, 0);
        }
        __syncthreads();
        for (int kk = 0; kk < N; ++kk) {
            const double *sk = scal + 4 * (kk & 1);
            const double tk = sk[0], sc = sk[1], beta = sk[2];
            const int part = tid / 80, jj = tid - part * 80, j = kk + 1 + jj;  // columns kk+1 .. N (N = innovation)
            const bool act = part < QP && j <= N;
            const int i0 = kk + 1 + part;                                    // rows i0, i0 + 3, ...
            if (tk != 0.0 && act) {
                // essential part v = tail / (c0 - beta) is formed on the fly: column kk itself is rewritten last
                const double *pv = RQ + i0 * ME_HS + kk, *pc = RQ + i0 * ME_HS + j;
                double t0 = 0.0, t1 = 0.0;
                int i = i0;
                for (; i + QP < mk; i += 2 * QP, pv += 2 * QP * ME_HS, pc += 2 * QP * ME_HS) {
                    t0 = fma(pv[0], pc[0], t0);
                    t1 = fma(pv[QP * ME_HS], pc[QP * ME_HS], t1);
                }
                if (i < mk) t0 = fma(pv[0], pc[0], t0);
                T3[part * 80 + jj] = t0 + t1;
                if (part == 0) T3[QP * 80 + jj] = RQ[kk * ME_HS + j];  // row kk is rewritten by part 0 below
            }
            __syncthreads();
            if (tk != 0.0 && act) {
                double dsum = 0.0;
#pragma unroll
                for (int q = 0; q < QP; ++q) dsum += T3[q * 80 + jj];
                const double tt = tk * fma(sc, dsum, T3[QP * 80 + jj]);
                const double ts = tt * sc;
                const double *pv = RQ + i0 * ME_HS + kk;
                double *pc = RQ + i0 * ME_HS + j;
                for (int i = i0; i < mk; i += QP, pv += QP * ME_HS, pc += QP * ME_HS) pc[0] = fma(-ts, pv[0], pc[0]);
                if (part == 0) RQ[kk * ME_HS + j] -= tt;
            }
            // partial norms of the next column's tail (rows > kk+1), by the three threads that have just updated it
            if (jj == 0 && part < QP && kk + 1 < N) {
                double t = 0.0;
                for (int i = i0 + (part == 0 ? QP : 0); i < mk; i += QP) {
                    const double v = RQ[i * ME_HS + kk + 1];
                    t = fma(v, v, t);
                }
                T3[(QP + 1) * 80 + part] = t;
            }
            __syncthreads();
            if (tk != 0.0) {
                for (int i = kk + 1 + tid; i < mk; i += MS_T) RQ[i * ME_HS + kk] *= sc;
            } else {
                for (int i = kk + 1 + tid; i < mk; i += MS_T) RQ[i * ME_HS + kk] = 0.0;
            }
            if (tid == 0) RQ[kk * ME_HS + kk] = beta;
            if (tid == 32 && kk + 1 < N)
                {
                double nsum = 0.0;
#pragma unroll
                for (int q = 0; q < QP; ++q) nsum += T3[(QP + 1) * 80 + q];
                reflector(RQ[(kk + 1) * ME_HS + kk + 1], nsum, scal + 4 * ((kk + 1) & 1), kk + 1);
            }
            __syncthreads();
        }
        if (tid < N) nu[tid] = RQ[tid * ME_HS + N];   // Q^T nu, first N entries (:811)
        // ---- thin Q = householderQ() * Identity(mk, N) into RH (:802-803): reflectors last to first; column j < kk of
        //      the partial product is still e_j, which reflector kk leaves alone ------------------------------------------
        for (int e = tid; e < mk * ME_HS; e += MS_T) {
            const int r = e / ME_HS, c = e - r * ME_HS;
            RH[e] = (r == c && c < N) ? 1.0 : 0.0;
        }
        __syncthreads();
        for (int kk = N - 1; kk >= 0; --kk) {
            const double tk = tau[kk];
            if (tk != 0.0) {   // uniform
                const int part = tid / 80, jj = tid - part * 80, j = kk + jj;
                const bool act = part < QP && j < N;
                const int i0 = kk + 1 + part;
                if (act) {
                    const double *pv = RQ + i0 * ME_HS + kk, *pc = RH + i0 * ME_HS + j;
                    double t0 = 0.0, t1 = 0.0;
                    int i = i0;
                    for (; i + QP < mk; i += 2 * QP, pv += 2 * QP * ME_HS, pc += 2 * QP * ME_HS) {
                        t0 = fma(pv[0], pc[0], t0);
                        t1 = fma(pv[QP * ME_HS], pc[QP * ME_HS], t1);
                    }
                    if (i < mk) t0 = fma(pv[0], pc[0], t0);
                    T3[part * 80 + jj] = t0 + t1;
                    if (part == 0) T3[QP * 80 + jj] = RH[kk * ME_HS + j];
                }
                __syncthreads();
                if (act) {
                    double dsum = 0.0;
#pragma unroll
                    for (int q = 0; q < QP; ++q) dsum += T3[q * 80 + jj];
                    const double tt = tk * (dsum + T3[QP * 80 + jj]);
                    const double *pv = RQ + i0 * ME_HS + kk;
                    double *pc = RH + i0 * ME_HS + j;
                    for (int i = i0; i < mk; i += QP, pv += QP * ME_HS, pc += QP * ME_HS) pc[0] = fma(-tt, pv[0], pc[0]);
                    if (part == 0) RH[kk * ME_HS + j] -= tt;
                }
                __syncthreads();
            }
        }
        // ---- Rr = Q^T R' Q (:814) into RS (packed lower).  A diagonal R (flagged once per launch by
        //      msckf_rdiag_kernel) makes R' Q a row scaling: Rr = sum_i r_i q_i q_i^T -----------------------------------------
        if (a.misc[0]) {
            if (tid < mk) wv[tid] = __ldg(a.R + (size_t)(compact ? kept[tid] : tid) * (M + 1));
            __syncthreads();
            for (int e = tid; e < NP; e += MS_T) {
                int r = (int)((sqrtf(8.0f * e + 1.0f) - 1.0f) * 0.5f);
                r += (tri(r + 1, 0) <= e) - (tri(r, 0) > e);
                const int c = e - tri(r, 0);
                double s0 = 0.0, s1 = 0.0;
                int i = 0;
                for (; i + 1 < mk; i += 2) {
                    s0 = fma(RH[i * ME_HS + r] * wv[i], RH[i * ME_HS + c], s0);
                    s1 = fma(RH[(i + 1) * ME_HS + r] * wv[i + 1], RH[(i + 1) * ME_HS + c], s1);
                }
                if (i < mk) s0 = fma(RH[i * ME_HS + r] * wv[i], RH[i * ME_HS + c], s0);
                RS[e] = s0 + s1;
            }
            __syncthreads();
        } else
        for (int b0 = 0; b0 < N; b0 += 8) {
            for (int e = tid; e < mk * 8; e += MS_T) {
                const int i = e >> 3, b = e & 7;
                const double *Rrow = a.R + (size_t)(compact ? kept[i] : i) * M;
                double sacc = 0.0;
                if (b0 + b < N)
                    for (int j = 0; j < mk; ++j) sacc = fma(__ldg(Rrow + (compact ? kept[j] : j)), RH[j * ME_HS + b0 + b], sacc);
                T3[e] = sacc;
            }
            __syncthreads();
            for (int e = tid; e < N * 8; e += MS_T) {
                const int r = e >> 3, c = b0 + (e & 7);
                if (c < N && c <= r) {
                    double sacc = 0.0;
                    for (int i = 0; i < mk; ++i) sacc = fma(RH[i * ME_HS + r], T3[i * 8 + (e & 7)], sacc);
                    RS[tri(r, c)] = sacc;
                }
            }
            __syncthreads();
        }
        // ---- covXZ = P Hr^T (N x N, row = state) into RH; Hr = upper triangle of RQ rows 0..N-1 (:808) --------------
        for (int e = tid; e < N * N; e += MS_T) {
            const int i = e / N, j = e - i * N;  // covXZ[j][i] = sum_{l >= i} Hr[i][l] P(l, j); a warp shares i (broadcast Hr)
            double sacc = 0.0;
            for (int l = i; l < N; ++l) sacc = fma(RQ[i * ME_HS + l], Psym(l, j), sacc);
            RH[j * ME_HS + i] = sacc;
        }
        __syncthreads();
        // ---- S = Hr covXZ + Rr (:330), packed lower in RS ---------------------------------------------------------
        for (int e = tid; e < NP; e += MS_T) {
            int r = (int)((sqrtf(8.0f * e + 1.0f) - 1.0f) * 0.5f);
            r += (tri(r + 1, 0) <= e) - (tri(r, 0) > e);
            const int c = e - tri(r, 0);
            double sacc = RS[e];
            for (int l = r; l < N; ++l) sacc = fma(RQ[r * ME_HS + l], RH[l * ME_HS + c], sacc);
            RS[e] = sacc;
        }
        __syncthreads();
        if (tid < mq) Yb[N * ys + tid] = nu[tid];
        chol_blocked(RS, N, flags, invd, PS, Yb, N, ys, Yb + N * ys);
        solved = true;
        if (!flags[0]) {
            if (tid == 0) a.status[inst] |= SLB_ST_CHOL_FAIL;
            continue;
        }
        }
        // ---- Y = covXZ Ls^-T: blocked right-looking TRSM, 8-column panels (thread per row), DMMA updates.  The innovation
        //      rides along as row N: [covXZ; nu^T] Ls^-T has w^T = (Ls^-1 nu)^T as its last row, so the forward substitution
        //      for w costs nothing extra (it used to be 100 sequential steps on one warp with the CTA waiting) ---------------
        //      When S had to be factored anew, chol_blocked has already carried these rows along; what follows is the
        //      stand-alone solve against the factor that the outlier gate left behind.
        const int nrt2 = (N + 8) >> 3;   // row tiles including row N
        for (int p0 = 0; p0 < (solved ? 0 : mq); p0 += 8) {
            const int pb = min(8, mq - p0);
            for (int i = tid; i <= N; i += MS_T) {
                double *row = Yb + i * ys + p0;
                double x[8];
#pragma unroll
                for (int c = 0; c < 8; ++c) {
                    if (c < pb) {
                        double sv = row[c];
#pragma unroll
                        for (int q = 0; q < 8; ++q)
                            if (q < c) sv = fma(-x[q], RS[tri(p0 + c, p0 + q)], sv);
                        x[c] = sv * invd[p0 + c];
                        row[c] = x[c];
                    }
                }
            }
            __syncthreads();
            const int j0 = p0 + pb, nct = (mq - j0 + 7) >> 3;
            for (int t = warp; t < nrt2 * nct; t += MS_W) {
                const int tr = t / nct, tc = t - tr * nct;
                const int ai = 8 * tr + fr, bj = j0 + 8 * tc + fr;
                double d0 = 0.0, d1 = 0.0;
                const double *pa = Yb + min(ai, N) * ys + p0 + fk, *pb2 = RS + tri(min(bj, mq - 1), p0) + fk;
                dmma884(d0, d1, pa[0], pb2[0]);
                dmma884(d0, d1, pa[4], pb2[4]);
                const int oc = j0 + 8 * tc + 2 * fk;
                if (ai <= N) {
                    if (oc < mq) Yb[ai * ys + oc] -= d0;
                    if (oc + 1 < mq) Yb[ai * ys + oc + 1] -= d1;
                }
            }
            __syncthreads();
        }
        // ---- delta = Y w (:337), w = row N of the solve ---------------------------------------------------------------
        for (int i = warp; i < N; i += MS_W) {
            double sacc = 0.0;
            const double *wrow = Yb + N * ys;
            for (int q = lane; q < mq; q += 32) sacc += Yb[i * ys + q] * wrow[q];
            sacc = warp_sum(sacc);
            if (lane == 0) dl[i] = sacc;
        }
        // ---- Pk -= K S K^T = Y Y^T (:336) straight to the HBM record: lower 8x8 tiles, K = mq ----------------------
        {
            const int ntiles = nrt * (nrt + 1) / 2;
            for (int t = warp; t < ntiles; t += MS_W) {
                int tr, tc;
                tri_tile(t, tr, tc);
                const int ai = 8 * tr + fr;
                const double *pa = Yb + min(ai, N - 1) * ys + fk, *pb = Yb + min(8 * tc + fr, N - 1) * ys + fk;
                double d0 = 0.0, d1 = 0.0;
                const int kfull = mq & ~3;   // mq is even: at most one ragged k-step
#pragma unroll 4
                for (int k0 = 0; k0 < kfull; k0 += 4) dmma884(d0, d1, pa[k0], pb[k0]);
                if (kfull < mq) {
                    const bool in = kfull + fk < mq;
                    dmma884(d0, d1, in ? pa[kfull] : 0.0, in ? pb[kfull] : 0.0);
                }
                const int r = ai, c = 8 * tc + 2 * fk;
                if (r < N) {
                    if (c <= r) Pg[tri(r, c)] = RA[tri(r, c)] - d0;
                    if (c + 1 <= r) Pg[tri(r, c + 1)] = RA[tri(r, c + 1)] - d1;
                }
            }
        }
        __syncthreads();
        // ---- mu = mu [+] K nu (:337), thread per block --------------------------------------------------------------
        bool finite = true;
        if (tid < NB) {
            const int b = tid, qo = ms_qoff(b);
            const double d[3] = {dl[3 * b], dl[3 * b + 1], dl[3 * b + 2]};
            if (ms_so3(b)) {
                double e[4], q[4];
                so3_exp(d, 1.0, e);
                quat_mul(mu + qo, e, q);
#pragma unroll
                for (int c = 0; c < 4; ++c) { mug[qo + c] = q[c]; finite = finite && isfinite(q[c]); }
            } else {
#pragma unroll
                for (int c = 0; c < 3; ++c) {
                    const double o = mu[qo + c] + d[c];
                    mug[qo + c] = o;
                    finite = finite && isfinite(o);
                }
            }
        }
        if (!finite) atomicOr(a.status + inst, SLB_ST_NONFINITE);
    }
}

}  // namespace slbd

namespace slb {

template <int PM, bool PIN>
static int launch_ms_predict_t(const FilterArgs &a, cudaStream_t s) {
    constexpr int WPB = 8;
    constexpr size_t smem = (size_t)WPB * slbd::PRED_SM * sizeof(double);
    auto kern = slbd::predict12_kernel<PM, WPB, 0, 0, false, PIN>;
    SLB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<(a.B + WPB - 1) / WPB, WPB * 32, smem, s>>>(a);
    count_launch();
    SLB_CUDA(cudaGetLastError());
    return SLB_OK;
}

int launch_msckf_predict(int pm, const FilterArgs &a, cudaStream_t s) {
    // a.qs != 0: per-instance Q (slb_set_noise_layout)
    if (pm == SLB_PM_MSCKF_DELTAPOSE)
        return a.qs ? launch_ms_predict_t<SLB_PM_MSCKF_DELTAPOSE, true>(a, s) : launch_ms_predict_t<SLB_PM_MSCKF_DELTAPOSE, false>(a, s);
    if (pm == SLB_PM_USCKF_TEST)
        return a.qs ? launch_ms_predict_t<SLB_PM_USCKF_TEST, true>(a, s) : launch_ms_predict_t<SLB_PM_USCKF_TEST, false>(a, s);
    return set_error(SLB_ERR_INVALID, "msckf: unsupported process model");
}

int launch_msckf_update(int mm, const FilterArgs &a, cudaStream_t s) {
    if (mm != SLB_MM_MSCKF_REPROJ) return set_error(SLB_ERR_INVALID, "msckf: unsupported measurement model");
    if (a.k < 1 || a.k > 10 || a.m > slbd::MS_MMAX || a.m < 2)
        return set_error(SLB_ERR_INVALID, "msckf update: needs 1..10 clones and 2 <= m <= 100");
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const size_t smem = (size_t)slbd::MS_SMEM_DOUBLES * sizeof(double);
    SLB_CUDA(cudaFuncSetAttribute(slbd::msckf_update_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int grid = a.B < sms ? a.B : sms;  // one persistent CTA per SM
    slbd::msckf_update_kernel<<<grid, slbd::MS_T, smem, s>>>(a);
    count_launch();
    SLB_CUDA(cudaGetLastError());
    return SLB_OK;
}

int launch_msckf_update_ekf(int mm, const FilterArgs &a, cudaStream_t s) {
    if (mm != SLB_MM_MSCKF_REPROJ) return set_error(SLB_ERR_INVALID, "msckf: unsupported measurement model");
    if (a.k < 1 || a.k > 10 || a.m > slbd::MS_MMAX || a.m < 2 || (a.m & 1))
        return set_error(SLB_ERR_INVALID, "msckf EKF update: needs 1..10 clones and an even 2 <= m <= 100");
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const size_t smem = (size_t)slbd::ME_SMEM_DOUBLES * sizeof(double);
    SLB_CUDA(cudaFuncSetAttribute(slbd::msckf_ekf_update_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int grid = a.B < sms ? a.B : sms;  // one persistent CTA per SM
    slbd::msckf_rdiag_kernel<<<1, 256, 0, s>>>(a.R, a.m, a.misc);
    slbd::msckf_ekf_update_kernel<<<grid, slbd::MS_T, smem, s>>>(a);
    count_launch(2);
    SLB_CUDA(cudaGetLastError());
    return SLB_OK;
}

}  // namespace slb

#ifdef SLB_MSCKF_PHASES
extern "C" int slb_debug_msckf_phases(long long *out) {
    return (int)cudaMemcpyFromSymbol(out, slbd::ms_phase_dbg, sizeof(long long) * 4 * 32);
}
#endif
#ifdef SLB_CHOL_TIMING
extern "C" int slb_debug_chol(long long *out) {
    return (int)cudaMemcpyFromSymbol(out, slbd::chol_dbg, sizeof(long long) * 16 * 16 * 8);
}
#endif
