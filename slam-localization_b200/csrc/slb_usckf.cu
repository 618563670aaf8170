// slb_usckf.cu -- localization::Usckf<AugmentedState,State>: predict, update, cloning,
// setMeasurement (src/filters/Usckf.hpp), one filter instance per WARP.
//
// Instance record in HBM: mu[qstride] (statek 13 | statek_l 13 | statek_i 13 | featuresk | featuresk_l)
// and the lower triangle of Pk as 8 x 8 tiles in DMMA accumulator order, P[prec(N, i, j)] (slb_math.cuh): off-diagonal
// tiles row-major, diagonal tiles packed lower, N(N+1)/2 doubles padded to 128 B.
// A record is contiguous, so a warp streams it with one TMA bulk copy (cp.async.bulk -> UBLKCP).
//
// predict (Usckf.hpp:113-244) touches only statek_i: rows 24..35, i.e. tile rows 3 and 4 (rows 24..39, one
//   contiguous span of 520 doubles at N >= 40), and the 12-wide segments of the feature rows below.  Called alone it is
//   predict12_kernel (slb_predict12.cuh), which fetches just those rows and runs predict12_block on them, the body the
//   fused step runs on its resident record.  Lane s evaluates sigma point s (25 of 32 lanes); Fk = Pxy^T Pii^-1 is
//   obtained as W^T L^-1 with W = 0.5 (dY+ - dY-) by a triangular solve, because X_i [-] mu_old is +-L e_j by
//   construction (same algebra as :152-154, without the explicit inverse).
// update (Usckf.hpp:260-308) and the fused predict+update step: slb_usckf_step.cuh (record resident in shared
//   memory, blocked square-root-free factorisation on DMMA accumulator tiles, sigma points streamed per 16 columns).
#include "slb_predict12.cuh"
#include "slb_usckf_step.cuh"

namespace slbd {

// =====================================================================================================
// cloning (Usckf.hpp:391-433) and setMeasurement (:322-389): pure data movement, thread per element
// =====================================================================================================
__global__ void usckf_clone_kernel(slb::FilterArgs a, int mode) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int per = 13 + 12 * 12 * 2;  // 13 mean scalars + two 12x12 blocks' worth of work items
    if (t >= (int64_t)a.B * per) return;
    const int inst = (int)(t / per), e = (int)(t - (int64_t)inst * per);
    double *P = a.P + (size_t)inst * a.pstride, *mu = a.mu + (size_t)inst * a.qstride;
    const int N = 36 + a.nk + a.nl;
    auto at = [&](int r, int c) -> double & { return P[prec(N, r, c)]; };   // r >= c
    auto sym = [&](int r, int c) { return r >= c ? at(r, c) : at(c, r); };
    if (e < 13) {
        if (mode == SLB_STATEK_I) mu[13 + e] = mu[26 + e];   // statek_l = statek_i (:401)
        else mu[e] = mu[13 + e];                              // statek = statek_l (:419)
        return;
    }
    const int q = e - 13, blk = q / 144, rc = q - blk * 144, r = rc / 12, c = rc - r * 12;
    if (mode == SLB_STATEK_I) {
        if (blk == 0) {
            // Pk+l = Pk+i (:405) and Pk+i|k+l = Pk+i (:406-407)
            const double v = sym(24 + r, 24 + c);
            if (c <= r) at(12 + r, 12 + c) = v;
            at(24 + r, 12 + c) = v;
        } else {
            // cross blocks with statek zeroed (:410-413)
            at(24 + r, c) = 0.0;
            at(12 + r, c) = 0.0;
        }
    } else if (blk == 0) {
        // Pk = Pk+l, Pk|k+l = Pk+l (:422-425)
        const double v = sym(12 + r, 12 + c);
        if (c <= r) at(r, c) = v;
        at(12 + r, c) = v;
    }
}
// The cloning kernel reads blocks other threads overwrite only in STATEK_I blk 0 (reads P_ii, writes
// P_ll / P_il) and STATEK_L blk 0 (reads P_ll, writes P_kk / P_lk): sources and destinations are disjoint.

__global__ void usckf_set_measurement_kernel(slb::FilterArgs a, int mode) {
    const int N = 36 + a.nk + a.nl;
    const int nfe = (N - 36) * N;  // rows 36..N-1 x all columns (entries above the diagonal do nothing)
    const int per = nfe + (mode == SLB_STATEK ? a.nk : a.nl);
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= (int64_t)a.B * per) return;
    const int inst = (int)(t / per), e = (int)(t - (int64_t)inst * per);
    double *P = a.P + (size_t)inst * a.pstride, *mu = a.mu + (size_t)inst * a.qstride;
    const int len = mode == SLB_STATEK ? a.nk : a.nl;
    const int f0 = mode == SLB_STATEK ? 0 : a.nk;  // first feature index being replaced
    if (e >= nfe) {
        const int c = e - nfe;
        mu[39 + f0 + c] = a.z[(size_t)inst * len + c];  // featuresk / featuresk_l = z (:335,:362)
        return;
    }
    const int r = 36 + e / N, c = e - (r - 36) * N;
    if (c > r) return;
    const int fr = r - 36, fc = c - 36;
    double v = 0.0;  // Pk.setZero() (:348,:376): every state<->feature and k<->k+l cross term
    if (c >= 36) {
        const bool rin = fr >= f0 && fr < f0 + len, cin = fc >= f0 && fc < f0 + len;
        if (rin && cin) v = a.R[(size_t)inst * a.rs + (fr - f0) * len + (fc - f0)];   // new block = R (:353,:381)
        else if (!rin && !cin) v = P[prec(N, r, c)];                // the block that stays (:355,:383)
    }
    P[prec(N, r, c)] = v;
}

}  // namespace slbd

namespace slb {

// the tiled record layout (prec) places every entry of the lower triangle once inside the N(N+1)/2 doubles of the
// packed one, and every off-diagonal tile row it holds starts on a 16-byte boundary
static constexpr bool prec_fills_record(int N) {
    bool seen[48 * 49 / 2] = {};
    for (int i = 0; i < N; ++i)
        for (int j = 0; j <= i; ++j) {
            const int o = slbd::prec(N, i, j);
            if (o < 0 || o >= N * (N + 1) / 2 || seen[o]) return false;
            if ((j & 7) == 0 && (j >> 3) < (i >> 3) && o % 2 != 0) return false;
            seen[o] = true;
        }
    return true;
}
#define SLB_USCKF_SHAPE(NK_, NL_) static_assert(prec_fills_record(36 + NK_ + NL_), "USCKF record layout");
SLB_USCKF_SHAPES(SLB_USCKF_SHAPE)
#undef SLB_USCKF_SHAPE

bool usckf_shape_supported(int nk, int nl) {
#define SLB_USCKF_SHAPE(NK_, NL_) \
    if (nk == NK_ && nl == NL_) return true;
    SLB_USCKF_SHAPES(SLB_USCKF_SHAPE)
#undef SLB_USCKF_SHAPE
    return false;
}

// record-resident kernel (slb_usckf_step.cuh): PRED && UPD = the fused step, UPD alone = update; PIN = per-instance noise,
// NIS = capture of the update's Mahalanobis distance
template <int NK, int NL, bool PRED, bool UPD, bool PIN, bool NIS = false>
static int launch_step_t(const FilterArgs &a, cudaStream_t s) {
    typedef slbd::StepCfg<NK, NL> C;
    // CTA shape: the register file (168 registers) holds 12 warps per SM.  Measured on the (3,9) fleet, 524 288 instances
    // (profiles/r02_usckf_cta_shape.txt): 1 / 2 / 3 / 4 / 6 / 12 warps per CTA = 6.37 / 6.94 / 6.06 / 6.19 / 5.77 / 6.53 ms per
    // step.  Two CTAs of six warps win: warps that start together walk the 104 KB unrolled instruction stream together
    // (the L1.5 instruction cache is 32 KB), while a single 12-warp CTA leaves the SM idle between its tail and the next
    // CTA's record loads.  Explicit CTA barriers to keep the warps aligned did not help (6.21 ms).
    // The PIN instantiation's RP extra doubles per warp (R staged next to z) fit in the slack of the same CTA shape for
    // every built shape: see the static_assert below.
    constexpr size_t pw = (size_t)(PIN ? C::SMP : C::SM) * sizeof(double);
    constexpr size_t SM_BYTES = 228 * 1024, RSV = 1024;
    constexpr int WPB = 2 * (6 * pw + RSV) <= SM_BYTES ? 6 : 4;
    constexpr size_t smem = (size_t)WPB * pw;
    constexpr int fit = (int)(SM_BYTES / (smem + RSV));
    constexpr int cap = 12 / WPB < 1 ? 1 : 12 / WPB;
    constexpr int MINB = fit > cap ? cap : fit < 1 ? 1 : fit;
    {   // per-instance noise must not cost the fused step a CTA
        constexpr size_t pw0 = (size_t)C::SM * sizeof(double);
        constexpr int WPB0 = 2 * (6 * pw0 + RSV) <= SM_BYTES ? 6 : 4;
        constexpr int fit0 = (int)(SM_BYTES / ((size_t)WPB0 * pw0 + RSV));
        static_assert(!PIN || (WPB == WPB0 && fit >= (fit0 < 12 / WPB0 ? fit0 : 12 / WPB0)), "PIN costs occupancy");
    }
    return launch(slbd::usckf_step_kernel<SLB_PM_USCKF_TEST, NK, NL, PRED, UPD, WPB, MINB, PIN, NIS>, (a.B + WPB - 1) / WPB,
                  WPB * 32, smem, s, a);
}

template <int NK, int NL, bool NIS>
static int launch_step_pin(bool predict, const FilterArgs &a, cudaStream_t s) {
    if ((predict && a.qs) || a.rs)
        return predict ? launch_step_t<NK, NL, true, true, true, NIS>(a, s) : launch_step_t<NK, NL, false, true, true, NIS>(a, s);
    return predict ? launch_step_t<NK, NL, true, true, false, NIS>(a, s) : launch_step_t<NK, NL, false, true, false, NIS>(a, s);
}
template <int NK, int NL>
static int launch_step_nknl(bool predict, const FilterArgs &a, cudaStream_t s) {
    return a.nis ? launch_step_pin<NK, NL, true>(predict, a, s) : launch_step_pin<NK, NL, false>(predict, a, s);
}

int launch_usckf(int pm, int mm, bool predict, bool update, const FilterArgs &a, cudaStream_t s) {
    if (predict && pm != SLB_PM_USCKF_TEST) return set_error(SLB_ERR_INVALID, "usckf: unsupported process model");
    if (update && mm != SLB_MM_USCKF_VO) return set_error(SLB_ERR_INVALID, "usckf: unsupported measurement model");
    // predict alone touches rows 24..35 of the record only: the partial-record kernel of slb_predict12.cuh
    if (predict && !update)
        return launch_predict12<SLB_PM_USCKF_TEST, 24, 26, true>(a, s);
    if (update) {
#define SLB_USCKF_SHAPE(NK_, NL_) \
    if (a.nk == NK_ && a.nl == NL_) return launch_step_nknl<NK_, NL_>(predict, a, s);
        SLB_USCKF_SHAPES(SLB_USCKF_SHAPE)
#undef SLB_USCKF_SHAPE
        return set_error(SLB_ERR_INVALID, "usckf update: (nk, nl) is not one of the built shapes (see slb_usckf_shape_supported)");
    }
    return SLB_OK;
}

int launch_usckf_clone(int mode, const FilterArgs &a, cudaStream_t s) {
    if (mode != SLB_STATEK_I && mode != SLB_STATEK_L) return SLB_OK;  // default: break (Usckf.hpp:428)
    const int64_t work = (int64_t)a.B * (13 + 288);
    return launch(slbd::usckf_clone_kernel, (unsigned)((work + 255) / 256), 256, 0, s, a, mode);
}

int launch_usckf_set_measurement(int mode, const FilterArgs &a, cudaStream_t s) {
    if (mode != SLB_STATEK && mode != SLB_STATEK_L) return SLB_OK;
    const int N = 36 + a.nk + a.nl;
    const int len = mode == SLB_STATEK ? a.nk : a.nl;
    if (len == 0) return SLB_OK;
    const int64_t work = (int64_t)a.B * ((N - 36) * N + len);
    return launch(slbd::usckf_set_measurement_kernel, (unsigned)((work + 255) / 256), 256, 0, s, a, mode);
}

}  // namespace slb
