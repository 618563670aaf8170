// slb_check.cu -- checkSigmaPoints() of localization::Usckf (Usckf.hpp:769-789) and localization::Msckf
// (Msckf.hpp:818-838): regenerate the sigma points of (mu_state, Pk), take their manifold mean muX and covariance
// Pktest = 0.5 sum (X_i [-] muX)(X_i [-] muX)^T and compare with (mu_state, Pk).  The reference asserts
// max|Pktest - Pk| <= 1e-6 and mu_state == muX; a batch reports both per instance instead of aborting.
//
// A diagnostic, not a hot path: one warp per instance, everything in shared memory (factor, accumulated covariance and
// the deviations of 32 sigma points at a time), plain FP64 SIMT.  It reuses no filter kernel on purpose -- it is the
// independent check of what those kernels assume (L L^T = Pk, [+] / [-] round trips, the weights of quirk Q1).
#include "slb_internal.h"
#include "slb_math.cuh"

namespace slbd {

SLB_DEV double warp_max(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

__global__ void __launch_bounds__(32) check_sigma_points_kernel(const double *mu, const double *P, int B, BatchLayout l,
                                                                int32_t *flags, double *diff) {
    extern __shared__ double sm[];
    const int lane = threadIdx.x;
    const int N = l.N, QD = l.QD, NP = l.NP, NS = 2 * N + 1;
    double *Lp = sm, *Pa = Lp + NP, *D = Pa + NP, *mus = D + 32 * N, *ref = mus + QD, *md = ref + QD;
    for (int inst = blockIdx.x; inst < B; inst += gridDim.x) {
        __syncwarp();
        for (int i = 0; i < N; ++i)
            for (int j = lane; j <= i; j += 32) { Lp[tri(i, j)] = P[l.P(inst, i, j)]; Pa[tri(i, j)] = 0.0; }
        for (int e = lane; e < QD; e += 32) { mus[e] = mu[l.mu(inst, e)]; ref[e] = mu[l.mu(inst, e)]; }
        __syncwarp();
        // ---- Eigen::LLT of Pk (lower triangle, Q8), right-looking, rows dealt to lanes -------------------------
        bool ok = true;
        for (int k = 0; k < N && ok; ++k) {
            const double dkk = Lp[tri(k, k)];
            ok = dkk > 0.0;
            if (!ok) break;
            const double s = sqrt(dkk), inv = 1.0 / s;
            __syncwarp();
            for (int i = k + lane; i < N; i += 32) Lp[tri(i, k)] = i == k ? s : Lp[tri(i, k)] * inv;
            __syncwarp();
            for (int i = k + 1 + lane; i < N; i += 32) {
                const double lik = Lp[tri(i, k)];
                for (int j = k + 1; j <= i; ++j) Lp[tri(i, j)] = fma(-lik, Lp[tri(j, k)], Lp[tri(i, j)]);
            }
            __syncwarp();
        }
        if (!ok) {
            if (lane == 0) {
                flags[inst] = 4;
                if (diff) { diff[2 * (size_t)inst] = 0.0; diff[2 * (size_t)inst + 1] = 0.0; }
            }
            continue;
        }
        // deviation of sigma point s from `ref`, written to row `lane` of D: X_s = mu [+] (+-L(:,j)), d = X_s [-] ref
        auto deviation = [&](int s) {
            double *d = D + lane * N;
            if (s >= NS) {
                for (int c = 0; c < N; ++c) d[c] = 0.0;
                return;
            }
            const int j = s >= 1 ? (s - 1) >> 1 : 0;
            const double sg = s == 0 ? 0.0 : (s & 1) ? 1.0 : -1.0;
            auto Lc = [&](int r) -> double { return r >= j ? sg * Lp[tri(r, j)] : 0.0; };
            int o = 0;
            for (int b = 0; b < l.nblk; ++b) {
                if ((l.so3mask >> b) & 1ull) {
                    const double v[3] = {Lc(3 * b), Lc(3 * b + 1), Lc(3 * b + 2)};
                    const double q[4] = {mus[o], mus[o + 1], mus[o + 2], mus[o + 3]};
                    const double r[4] = {ref[o], ref[o + 1], ref[o + 2], ref[o + 3]};
                    double e[4], x[4], t[4], w[3];
                    so3_exp(v, 1.0, e);
                    quat_mul(q, e, x);
                    quat_cmul(r, x, t);
                    so3_log(t, w);
                    d[3 * b] = w[0]; d[3 * b + 1] = w[1]; d[3 * b + 2] = w[2];
                    o += 4;
                } else {
                    for (int c = 0; c < 3; ++c) d[3 * b + c] = (mus[o + c] + Lc(3 * b + c)) - ref[o + c];
                    o += 3;
                }
            }
            for (int f = 0; f < l.nfeat; ++f) d[3 * l.nblk + f] = (mus[o + f] + Lc(3 * l.nblk + f)) - ref[o + f];
        };
        // ---- manifold mean (Usckf.hpp:601-627): start at X0, do { ref = ref [+] mean(X_i [-] ref) } while |.| > 1e-6 --
        int it = 0;
        double nrm2;
        do {
            for (int c = lane; c < N; c += 32) md[c] = 0.0;
            for (int s0 = 0; s0 < NS; s0 += 32) {
                __syncwarp();
                deviation(s0 + lane);
                __syncwarp();
                for (int c = lane; c < N; c += 32) {
                    double a = 0.0;
                    for (int t = 0; t < 32; ++t) a += D[t * N + c];
                    md[c] += a;
                }
            }
            __syncwarp();
            double part = 0.0;
            for (int c = lane; c < N; c += 32) {
                const double m = md[c] / (double)NS;
                md[c] = m;
                part += m * m;
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
            nrm2 = part;
            __syncwarp();
            // ref = ref [+] md, one block (or one feature scalar) per lane
            {
                int o = 0;
                for (int b = 0; b < l.nblk; ++b) {
                    const bool so3 = (l.so3mask >> b) & 1ull;
                    if (b % 32 == lane) {
                        if (so3) {
                            const double v[3] = {md[3 * b], md[3 * b + 1], md[3 * b + 2]};
                            const double q[4] = {ref[o], ref[o + 1], ref[o + 2], ref[o + 3]};
                            double e[4], x[4];
                            so3_exp(v, 1.0, e);
                            quat_mul(q, e, x);
                            for (int c = 0; c < 4; ++c) ref[o + c] = x[c];
                        } else {
                            for (int c = 0; c < 3; ++c) ref[o + c] += md[3 * b + c];
                        }
                    }
                    o += so3 ? 4 : 3;
                }
                for (int f = lane; f < l.nfeat; f += 32) ref[o + f] += md[3 * l.nblk + f];
            }
            __syncwarp();
        } while (sqrt(nrm2) > 1e-6 && ++it < 10000);
        // ---- Pktest = 0.5 sum (X_i [-] muX)(X_i [-] muX)^T, 32 sigma points at a time ---------------------------------
        for (int s0 = 0; s0 < NS; s0 += 32) {
            __syncwarp();
            deviation(s0 + lane);
            __syncwarp();
            for (int i = 0; i < N; ++i)
                for (int j = lane; j <= i; j += 32) {
                    double a = 0.0;
                    for (int t = 0; t < 32; ++t) a = fma(D[t * N + i], D[t * N + j], a);
                    Pa[tri(i, j)] += 0.5 * a;
                }
        }
        __syncwarp();
        double dP = 0.0;
        for (int i = 0; i < N; ++i)
            for (int j = lane; j <= i; j += 32) dP = fmax(dP, fabs(Pa[tri(i, j)] - P[l.P(inst, i, j)]));
        dP = warp_max(dP);
        // |muX [-] mu|_inf: ref [-] mus, block per lane
        double dm = 0.0;
        {
            int o = 0;
            for (int b = 0; b < l.nblk; ++b) {
                const bool so3 = (l.so3mask >> b) & 1ull;
                if (b % 32 == lane) {
                    if (so3) {
                        const double q[4] = {mus[o], mus[o + 1], mus[o + 2], mus[o + 3]};
                        const double r[4] = {ref[o], ref[o + 1], ref[o + 2], ref[o + 3]};
                        double t[4], w[3];
                        quat_cmul(q, r, t);
                        so3_log(t, w);
                        for (int c = 0; c < 3; ++c) dm = fmax(dm, fabs(w[c]));
                    } else {
                        for (int c = 0; c < 3; ++c) dm = fmax(dm, fabs(ref[o + c] - mus[o + c]));
                    }
                }
                o += so3 ? 4 : 3;
            }
            for (int f = lane; f < l.nfeat; f += 32) dm = fmax(dm, fabs(ref[o + f] - mus[o + f]));
        }
        dm = warp_max(dm);
        if (lane == 0) {
            // (!(x <= tol) also flags NaN)
            flags[inst] = (!(dP <= 1e-6) ? 1 : 0) | (!(dm <= 1e-12) ? 2 : 0);
            if (diff) { diff[2 * (size_t)inst] = dP; diff[2 * (size_t)inst + 1] = dm; }
        }
    }
}

}  // namespace slbd

namespace slb {

int launch_check_sigma_points(const slb_batch_s *h, int32_t *flags, double *diff, cudaStream_t s) {
    const slbd::BatchLayout &l = h->L;
    const size_t smem = ((size_t)2 * l.NP + 32 * l.N + 2 * l.QD + l.N) * sizeof(double);
    SLB_CUDA(cudaFuncSetAttribute(slbd::check_sigma_points_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int grid = h->B < 148 * 3 * 8 ? h->B : 148 * 3 * 8;
    slbd::check_sigma_points_kernel<<<grid, 32, smem, s>>>(h->mu, h->P, h->B, l, flags, diff);
    count_launch();
    SLB_CUDA(cudaGetLastError());
    return SLB_OK;
}

}  // namespace slb
