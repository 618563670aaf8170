// slb_consistency.cu -- filter consistency of a batch: NEES = e^T P_sub^-1 e with e = truth [-] mu over the tangent
// coordinates [t0, t0 + n), and the fleet sums of NEES and of the NIS the last update captured (slb_set_nis_capture).
//
// One warp per instance.  The marginal covariance P_sub = P[t0:t0+n, t0:t0+n] (lower triangle, read through the batch's
// BatchLayout, so SoA, tiled and packed records share the kernel) is staged packed in shared memory with e appended as
// row n: a right-looking Cholesky of that bordered matrix leaves L in rows 0..n-1 and y = L^-1 e (the forward
// substitution) in row n, so NEES = |y|^2 without an explicit inverse.  At the MSCKF's N = 72 the bordered triangle is
// 73 * 74 / 2 doubles = 21.6 KB per warp.  Each instance's result depends on its own data only (fixed lane roles, fixed
// reduction order); the fleet sums are FP64 atomics, one set per CTA.
#include "slb_internal.h"
#include "slb_math.cuh"
#include "slb_ptx.cuh"

namespace slbd {

constexpr int CONS_WPB = 8;

// tangent coordinate t of truth [-] mu for instance i (MTK: log(mu_q^-1 truth_q) on SO3 blocks, a difference elsewhere)
SLB_DEV double tangent_error(const double *mu, const double *truth, const BatchLayout &L, int i, int t) {
    const double *tr = truth + (size_t)i * L.QD;
    const int nb3 = 3 * L.nblk;
    if (t >= nb3) {
        const int c = nb3 + __popcll(L.so3mask) + (t - nb3);
        return tr[c] - mu[L.mu(i, c)];
    }
    const int b = t / 3, k = t - 3 * b;
    const int o = 3 * b + __popcll(L.so3mask & ((1ull << b) - 1ull));
    if ((L.so3mask >> b) & 1ull) {
        const double qm[4] = {mu[L.mu(i, o)], mu[L.mu(i, o + 1)], mu[L.mu(i, o + 2)], mu[L.mu(i, o + 3)]};
        double r[4], v[3];
        quat_cmul(qm, tr + o, r);
        so3_log(r, v);
        return k == 0 ? v[0] : k == 1 ? v[1] : v[2];   // (a runtime index would put v in local memory)
    }
    return tr[o + k] - mu[L.mu(i, o + k)];
}

__global__ void __launch_bounds__(CONS_WPB * 32) consistency_kernel(const double *mu, const double *P, const double *nis, int B,
                                                                    BatchLayout L, const double *truth, int t0, int n,
                                                                    double *nees, double *out) {
    extern __shared__ double sm[];
    __shared__ double red[CONS_WPB][6];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int W = ((n + 1) * (n + 2) / 2 + 1) / 2 * 2;   // bordered packed triangle, per warp
    double *A = sm + (size_t)warp * W;
    double acc[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};   // lane 0: NEES count, sum, sum of squares, then the same for NIS
    const double NaN = __longlong_as_double(0x7ff8000000000000ll);
    for (int i = blockIdx.x * CONS_WPB + warp; i < B; i += gridDim.x * CONS_WPB) {
        if (nis && lane == 0) {
            const double v = nis[i];
            if (isfinite(v)) { acc[3] += 1.0; acc[4] += v; acc[5] = fma(v, v, acc[5]); }
        }
        if (!truth) continue;
        __syncwarp();
        for (int r = 0; r < n; ++r)
            for (int c = lane; c <= r; c += 32) A[tri(r, c)] = P[L.P(i, t0 + r, t0 + c)];
        bool fin = true;
        for (int k = lane; k < n; k += 32) {
            const double e = tangent_error(mu, truth, L, i, t0 + k);
            fin = fin && isfinite(e);
            A[tri(n, k)] = e;
        }
        bool ok = __all_sync(FULL, fin);
        __syncwarp();
        // Cholesky of the bordered matrix, columns 0..n-1 (row n is e: it becomes L^-1 e)
        for (int k = 0; k < n && ok; ++k) {
            const double d = A[tri(k, k)];
            ok = d > 0.0 && d < INFINITY;
            if (!ok) break;
            const double inv = 1.0 / sqrt(d);
            __syncwarp();
            for (int r = k + 1 + lane; r <= n; r += 32) A[tri(r, k)] *= inv;
            __syncwarp();
            for (int r = k + 1 + lane; r <= n; r += 32) {
                const double lrk = A[tri(r, k)];
                const int cmax = r < n ? r : n - 1;
                for (int c = k + 1; c <= cmax; ++c) A[tri(r, c)] = fma(-lrk, A[tri(c, k)], A[tri(r, c)]);
            }
            __syncwarp();
        }
        double y2 = 0.0;
        if (ok)
            for (int k = lane; k < n; k += 32) y2 = fma(A[tri(n, k)], A[tri(n, k)], y2);
        y2 = warp_sum(y2);
        ok = ok && isfinite(y2);
        if (lane == 0) {
            if (nees) nees[i] = ok ? y2 : NaN;
            if (ok) { acc[0] += 1.0; acc[1] += y2; acc[2] = fma(y2, y2, acc[2]); }
        }
    }
    if (lane == 0)
#pragma unroll
        for (int k = 0; k < 6; ++k) red[warp][k] = acc[k];
    __syncthreads();
    if (threadIdx.x < 6) {
        double s = 0.0;
#pragma unroll
        for (int w = 0; w < CONS_WPB; ++w) s += red[w][threadIdx.x];
        if (s != 0.0) atomicAdd(out + threadIdx.x, s);
    }
}

}  // namespace slbd

namespace slb {

int launch_consistency(const slb_batch_s *h, const double *truth, int t0, int n, double *nees, double *out, cudaStream_t s) {
    const size_t smem = truth ? (size_t)slbd::CONS_WPB * (((n + 1) * (n + 2) / 2 + 1) / 2 * 2) * sizeof(double) : 0;
    auto kern = slbd::consistency_kernel;
    SLB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int dev = 0, sms = 148, per_sm = 1;
    SLB_CUDA(cudaGetDevice(&dev));
    SLB_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    SLB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, slbd::CONS_WPB * 32, smem));
    const int need = (h->B + slbd::CONS_WPB - 1) / slbd::CONS_WPB;
    const int cap = sms * (per_sm < 1 ? 1 : per_sm);
    kern<<<need < cap ? need : cap, slbd::CONS_WPB * 32, smem, s>>>(h->mu, h->P, h->nis, h->B, h->L, truth, t0, n, nees, out);
    count_launch();
    SLB_CUDA(cudaGetLastError());
    return SLB_OK;
}

}  // namespace slb
