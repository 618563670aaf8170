// slb_api.cu -- the extern "C" surface declared in include/slb.h: batch lifetime, host<->device
// state transfer (layout conversion kernels), dispatch to the filter kernels, diagnostics.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <atomic>
#include <new>

#include <dlfcn.h>
#include <nccl.h>

#include "slb_internal.h"
#include "slb_math.cuh"

namespace slb {

static thread_local char g_err[512] = "";
static std::atomic<int64_t> g_launches{0};

int set_error(int code, const char *what, cudaError_t ce) {
    if (ce != cudaSuccess)
        snprintf(g_err, sizeof(g_err), "%s: %s", what, cudaGetErrorString(ce));
    else
        snprintf(g_err, sizeof(g_err), "%s", what);
    return code;
}
void count_launch(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); }

// ---- layout conversion kernels: dense instance-major host arrays <-> the batch (h->L) ---------------------------
// Means: thread t = (instance, scalar), scalar fastest.  mu_in stores instances [b0, b0 + cnt); mu_out loads the slice
// [off, off + len) of their q-vectors.
__global__ void mu_in(const double *src, double *mu, slbd::BatchLayout L, int b0, int cnt) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= cnt * L.QD) return;
    const int i = t / L.QD, c = t - i * L.QD;
    mu[L.mu(b0 + i, c)] = src[t];
}
__global__ void mu_out(const double *mu, double *dst, slbd::BatchLayout L, int b0, int cnt, int off, int len) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= cnt * len) return;
    const int i = t / len, c = t - i * len;
    dst[t] = mu[L.mu(b0 + i, off + c)];
}
// thread t of a launch over `per` entries of each of `cnt` instances -> (instance i, entry k): the instance fastest
// for SoA, the entry fastest for records, so that consecutive threads store to consecutive doubles of the batch
SLB_DEV void split(const slbd::BatchLayout &L, int64_t t, int cnt, int per, int &i, int &k) {
    if (L.soa) { k = (int)(t / cnt); i = (int)(t - (int64_t)k * cnt); }
    else { i = (int)(t / per); k = (int)(t - (int64_t)i * per); }
}
// (r, c), r >= c, of packed lower-triangle entry e
SLB_DEV void tri_rc(int e, int &r, int &c) {
    r = (int)((sqrt(8.0 * e + 1.0) - 1.0) * 0.5);
    while (r * (r + 1) / 2 > e) --r;
    while ((r + 1) * (r + 2) / 2 <= e) ++r;
    c = e - r * (r + 1) / 2;
}
// Covariances: the lower triangle of dense src goes to the batch; P_out writes both triangles of dense dst.
__global__ void P_in(const double *src, double *P, slbd::BatchLayout L, int b0, int cnt) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= (int64_t)cnt * L.NP) return;
    int i, e, r, c;
    split(L, t, cnt, L.NP, i, e);
    tri_rc(e, r, c);
    P[L.P(b0 + i, r, c)] = src[((size_t)i * L.N + r) * L.N + c];
}
__global__ void P_out(const double *P, double *dst, slbd::BatchLayout L, int b0, int cnt) {
    const int N = L.N;
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= (int64_t)cnt * N * N) return;
    const int i = (int)(t / (N * N)), rc = (int)(t - (int64_t)i * N * N);
    int r = rc / N, c = rc - r * N;
    if (c > r) { const int x = r; r = c; c = x; }
    dst[t] = P[L.P(b0 + i, r, c)];
}

// fleet initialisation: instance i <- instance i % count (Monte-Carlo replicas of `count` priors), the means (a = mu)
// or the covariances (cov, a = P)
__global__ void replicate(double *a, slbd::BatchLayout L, int B, int count, bool cov) {
    const int per = cov ? L.NP : L.QD;
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= (int64_t)per * B) return;
    int i, k;
    split(L, t, B, per, i, k);
    if (i < count) return;
    if (cov) {
        int r, c;
        tri_rc(k, r, c);
        a[L.P(i, r, c)] = a[L.P(i % count, r, c)];
    } else {
        a[L.mu(i, k)] = a[L.mu(i % count, k)];
    }
}

__global__ void status_count(const int32_t *st, int B, unsigned long long *counts) {
    unsigned long long c[SLB_NSTATUS];
#pragma unroll
    for (int b = 0; b < SLB_NSTATUS; ++b) c[b] = 0;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < B; i += gridDim.x * blockDim.x) {
        const int s = st[i];
#pragma unroll
        for (int b = 0; b < SLB_NSTATUS; ++b) c[b] += (s >> b) & 1;
    }
#pragma unroll
    for (int b = 0; b < SLB_NSTATUS; ++b) {
        for (int o = 16; o > 0; o >>= 1) c[b] += __shfl_down_sync(0xffffffffu, c[b], o);
        if ((threadIdx.x & 31) == 0 && c[b]) atomicAdd(counts + b, c[b]);
    }
}

// Ensemble statistics: out = {count, sum x, sum x x^T}, x = vectorised mean (log of SO3 blocks).
// Persistent CTAs, chunks of 64 instances staged in shared memory, register accumulators.
constexpr int STAT_CHUNK = 64, STAT_TPB = 256, STAT_MAXACC = 24;
__global__ void __launch_bounds__(STAT_TPB) ensemble_stats_kernel(const double *mu, int B, slbd::BatchLayout L, double *out) {
    extern __shared__ double xs[];  // [STAT_CHUNK][N]
    const int N = L.N;
    const int nent = N * N + N;
    double acc[STAT_MAXACC];
#pragma unroll
    for (int k = 0; k < STAT_MAXACC; ++k) acc[k] = 0.0;
    const int nchunks = (B + STAT_CHUNK - 1) / STAT_CHUNK;
    for (int ch = blockIdx.x; ch < nchunks; ch += gridDim.x) {
        const int base = ch * STAT_CHUNK;
        const int cnt = min(STAT_CHUNK, B - base);
        __syncthreads();
        if ((int)threadIdx.x < cnt) {
            const int i = base + threadIdx.x;
            double *x = xs + threadIdx.x * N;
            int o = 0;
            for (int b = 0; b < L.nblk; ++b) {
                if ((L.so3mask >> b) & 1ull) {
                    const double q[4] = {mu[L.mu(i, o)], mu[L.mu(i, o + 1)], mu[L.mu(i, o + 2)], mu[L.mu(i, o + 3)]};
                    double v[3];
                    slbd::so3_log(q, v);
                    x[3 * b] = v[0]; x[3 * b + 1] = v[1]; x[3 * b + 2] = v[2];
                    o += 4;
                } else {
                    x[3 * b] = mu[L.mu(i, o)]; x[3 * b + 1] = mu[L.mu(i, o + 1)]; x[3 * b + 2] = mu[L.mu(i, o + 2)];
                    o += 3;
                }
            }
            for (int f = 0; f < L.nfeat; ++f) x[3 * L.nblk + f] = mu[L.mu(i, o + f)];
        }
        __syncthreads();
#pragma unroll
        for (int k = 0; k < STAT_MAXACC; ++k) {
            const int e = threadIdx.x + k * STAT_TPB;
            if (e < nent) {
                double s = 0.0;
                if (e < N) {
                    for (int t = 0; t < cnt; ++t) s += xs[t * N + e];
                } else {
                    const int r = (e - N) / N, c = (e - N) - r * N;
                    for (int t = 0; t < cnt; ++t) s += xs[t * N + r] * xs[t * N + c];
                }
                acc[k] += s;
            }
        }
    }
#pragma unroll
    for (int k = 0; k < STAT_MAXACC; ++k) {
        const int e = threadIdx.x + k * STAT_TPB;
        if (e < nent && acc[k] != 0.0) atomicAdd(out + 1 + e, acc[k]);
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) atomicAdd(out, (double)B);
}

// FP64 FMA-rate microbenchmark (roofline denominator for the FP64-bound configs; not in
// MEASURED_PEAKS.json).  16 independent DFMA chains per thread, every SM saturated.
__global__ void __launch_bounds__(256) fp64_peak_kernel(double *sink, int iters, double a, double b) {
    double x[16];
#pragma unroll
    for (int k = 0; k < 16; ++k) x[k] = a + k + threadIdx.x;
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int k = 0; k < 16; ++k) x[k] = fma(x[k], b, a);
    }
    double s = 0;
#pragma unroll
    for (int k = 0; k < 16; ++k) s += x[k];
    if (s == 12345.678) sink[0] = s;
}

static cudaStream_t S(void *p) { return (cudaStream_t)p; }

static FilterArgs make_args(slb_handle h) {
    FilterArgs a;
    memset(&a, 0, sizeof(a));
    a.mu = h->mu; a.P = h->P; a.status = h->status; a.outliers = h->outliers;
    a.B = h->B; a.stride = h->L.stride; a.pstride = h->L.pstride; a.qstride = h->L.qstride;
    a.nk = h->cfg.nk; a.nl = h->cfg.nl; a.k = h->cfg.nclones;
    a.misc = h->misc_dev;
    a.out_off = h->out_off; a.out_len = h->out_len;
    a.nis = h->nis;
    return a;
}

static int pm_nu(int pm) { return pm == SLB_PM_MSCKF_DELTAPOSE ? 13 : 6; }

// The storage of a batch of B instances of a configuration slb_create accepted (DESIGN §3)
static constexpr slbd::BatchLayout batch_layout(int kind, int layout, int nk, int nl, int nclones, int B) {
    slbd::BatchLayout L{};
    switch (kind) {
        case SLB_KIND_UKF:  // pos, orient [, vel]
            L.N = layout; L.QD = layout + 1;
            L.nblk = layout / 3; L.so3mask = 0x2;
            break;
        case SLB_KIND_USCKF:  // statek | statek_l | statek_i (pos, orient, velo, angvelo each), featuresk | featuresk_l
            L.N = 36 + nk + nl; L.QD = 39 + nk + nl;
            L.nblk = 12; L.so3mask = 0x222; L.nfeat = nk + nl;
            break;
        default:  // MSCKF: pos, orient, velo, angvelo, then (pos, orient) per clone
            L.N = 12 + 6 * nclones; L.QD = 13 + 7 * nclones;
            L.nblk = 4 + 2 * nclones; L.so3mask = 0x2;
            for (int j = 0; j < nclones; ++j) L.so3mask |= 1ull << (4 + 2 * j + 1);
    }
    L.NP = L.N * (L.N + 1) / 2;
    L.soa = kind == SLB_KIND_UKF;
    L.tiled = kind == SLB_KIND_USCKF;
    L.stride = (B + 31) / 32 * 32;
    L.pstride = (L.NP + 15) / 16 * 16;
    L.qstride = (L.QD + 1) / 2 * 2;
    return L;
}
// P(i, ., .) puts the NP entries of each instance on distinct doubles inside the P_size(B) of the batch, a record's in
// its first NP: with B = 32 a SoA batch is filled without a gap, a record up to its padding
static constexpr bool P_fills_storage(const slbd::BatchLayout &L, int B) {
    bool seen[8192] = {};
    if (L.P_size(B) > 8192) return false;
    for (int i = 0; i < B; ++i)
        for (int r = 0; r < L.N; ++r)
            for (int c = 0; c <= r; ++c) {
                const size_t o = L.P(i, r, c);
                if (o >= L.P_size(B) || seen[o]) return false;
                if (!L.soa && (o < (size_t)i * L.pstride || o >= (size_t)i * L.pstride + L.NP)) return false;
                seen[o] = true;
            }
    return true;
}
static_assert(P_fills_storage(batch_layout(SLB_KIND_UKF, SLB_LAYOUT_POSE6, 0, 0, 0, 32), 32), "UKF POSE6 storage");
static_assert(P_fills_storage(batch_layout(SLB_KIND_UKF, SLB_LAYOUT_MTK9, 0, 0, 0, 32), 32), "UKF MTK9 storage");
static_assert(P_fills_storage(batch_layout(SLB_KIND_MSCKF, 0, 0, 0, 10, 2), 2), "MSCKF storage");
#define SLB_USCKF_SHAPE(NK_, NL_) \
    static_assert(P_fills_storage(batch_layout(SLB_KIND_USCKF, 0, NK_, NL_, 0, 2), 2), "USCKF storage");
SLB_USCKF_SHAPES(SLB_USCKF_SHAPE)
#undef SLB_USCKF_SHAPE

}  // namespace slb

using namespace slb;

extern "C" {

int slb_version(void) { return SLB_VERSION; }
const char *slb_last_error(void) { return g_err; }
int64_t slb_launch_count(void) { return g_launches.load(); }

int slb_create(const slb_config *cfg, slb_handle *out) {
    if (!cfg || !out) return set_error(SLB_ERR_INVALID, "slb_create: null argument");
    *out = nullptr;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        return set_error(SLB_ERR_NO_DEVICE, "slb_create: no CUDA device (this engine has no CPU fallback)");
    }
    if (cfg->device < 0 || cfg->device >= ndev) return set_error(SLB_ERR_INVALID, "slb_create: bad device ordinal");
    if (cfg->batch <= 0) return set_error(SLB_ERR_INVALID, "slb_create: batch must be positive");
    DeviceGuard guard(cfg->device);  // no lasting side effect on the caller's current device
    {
        int cur = -1;
        if (cudaGetDevice(&cur) != cudaSuccess || cur != cfg->device) return set_error(SLB_ERR_CUDA, "slb_create: cudaSetDevice failed");
    }
    switch (cfg->kind) {
        case SLB_KIND_UKF:
            if (cfg->layout != SLB_LAYOUT_POSE6 && cfg->layout != SLB_LAYOUT_MTK9)
                return set_error(SLB_ERR_INVALID, "slb_create: UKF layout must be POSE6 or MTK9");
            break;
        case SLB_KIND_USCKF:
            if (!usckf_shape_supported(cfg->nk, cfg->nl))
                return set_error(SLB_ERR_INVALID,
                                 "slb_create: USCKF batches are built for nk in {3,6,9}, nl in {0,3,6,9} with nk + nl <= 12");
            break;
        case SLB_KIND_MSCKF:
            if (cfg->nclones < 0 || cfg->nclones > 10) return set_error(SLB_ERR_INVALID, "slb_create: MSCKF supports 0..10 clones");
            break;
        default:
            return set_error(SLB_ERR_INVALID, "slb_create: unknown kind");
    }
    slb_batch_s *h = new (std::nothrow) slb_batch_s();
    if (!h) return set_error(SLB_ERR_ALLOC, "slb_create: host allocation failed");
    memset(h, 0, sizeof(*h));
    h->cfg = *cfg;
    h->B = cfg->batch;
    h->L = batch_layout(cfg->kind, cfg->layout, cfg->nk, cfg->nl, cfg->nclones, cfg->batch);
    const slbd::BatchLayout &L = h->L;
    h->out_off = 0;
    h->out_len = L.QD;
    const size_t mu_bytes = L.mu_size(h->B) * 8, P_bytes = L.P_size(h->B) * 8;
    h->stage_bytes = (size_t)64 << 20;
    const size_t one = (size_t)L.N * L.N * 8;
    if (h->stage_bytes < one * 32) h->stage_bytes = one * 32;
    // the *_step_host entry points stage u | z | mu_out for the whole batch
    const size_t io = (size_t)h->B * (L.QD + 16 + (cfg->kind == SLB_KIND_MSCKF ? 104 : 4)) * 8;
    if (h->stage_bytes < io) h->stage_bytes = io;
    cudaError_t e = cudaSuccess;
    if (e == cudaSuccess) e = cudaMalloc(&h->mu, mu_bytes);
    if (e == cudaSuccess) e = cudaMalloc(&h->P, P_bytes);
    if (e == cudaSuccess) e = cudaMalloc(&h->status, (size_t)h->B * 4);
    if (e == cudaSuccess) e = cudaMalloc(&h->outliers, (size_t)h->B * 4);
    if (e == cudaSuccess) e = cudaMalloc(&h->stage, h->stage_bytes);
    if (e == cudaSuccess) e = cudaMalloc(&h->shared_small, 128 * 1024);
    if (e == cudaSuccess) e = cudaMalloc(&h->counts_dev, 8 * sizeof(int64_t));
    if (e == cudaSuccess) e = cudaMalloc(&h->misc_dev, 16 * sizeof(int32_t));
    for (int i = 0; i < SLB_NXS && e == cudaSuccess; ++i) {
        e = cudaStreamCreateWithFlags(&h->xs[i], cudaStreamNonBlocking);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&h->ev_done[i], cudaEventDisableTiming);
    }
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&h->ev_start, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&h->cap_stream, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaMemset(h->mu, 0, mu_bytes);
    if (e == cudaSuccess) e = cudaMemset(h->P, 0, P_bytes);
    if (e == cudaSuccess) e = cudaMemset(h->status, 0, (size_t)h->B * 4);
    if (e == cudaSuccess) e = cudaMemset(h->outliers, 0, (size_t)h->B * 4);
    if (e != cudaSuccess) {
        slb_destroy(h);
        return set_error(SLB_ERR_ALLOC, "slb_create: device allocation failed", e);
    }
    *out = h;
    return SLB_OK;
}

int slb_destroy(slb_handle h) {
    if (!h) return SLB_OK;
    DeviceGuard guard(h->cfg.device);
    cudaFree(h->mu); cudaFree(h->P); cudaFree(h->status); cudaFree(h->outliers);
    cudaFree(h->stage); cudaFree(h->shared_small); cudaFree(h->counts_dev); cudaFree(h->misc_dev); cudaFree(h->nis);
    for (int i = 0; i < SLB_NXS; ++i) {
        if (h->xs[i]) cudaStreamDestroy(h->xs[i]);
        if (h->ev_done[i]) cudaEventDestroy(h->ev_done[i]);
    }
    if (h->ev_start) cudaEventDestroy(h->ev_start);
    if (h->step_exec) cudaGraphExecDestroy(h->step_exec);
    if (h->cap_stream) cudaStreamDestroy(h->cap_stream);
    delete h;
    return SLB_OK;
}

int slb_set_output_slice(slb_handle h, int offset, int count) {
    if (!h || offset < 0 || count < 1 || offset + count > h->L.QD)
        return set_error(SLB_ERR_INVALID, "slb_set_output_slice: the slice must lie inside the q-vector");
    h->out_off = offset;
    h->out_len = count;
    return SLB_OK;
}
int slb_set_noise_layout(slb_handle h, int flags) {
    if (!h) return set_error(SLB_ERR_INVALID, "slb_set_noise_layout: null handle");
    if (flags < 0 || flags > (SLB_NOISE_Q_PER_INSTANCE | SLB_NOISE_R_PER_INSTANCE))
        return set_error(SLB_ERR_INVALID, "slb_set_noise_layout: flags must be a combination of SLB_NOISE_Q_PER_INSTANCE and "
                                          "SLB_NOISE_R_PER_INSTANCE");
    if (h->cfg.kind == SLB_KIND_MSCKF && (flags & SLB_NOISE_R_PER_INSTANCE))
        return set_error(SLB_ERR_INVALID, "slb_set_noise_layout: MSCKF update noise is shared by the batch (only Q may be per instance)");
    h->noise = flags;
    return SLB_OK;
}
int slb_set_nis_capture(slb_handle h, int on) {
    if (!h) return set_error(SLB_ERR_INVALID, "slb_set_nis_capture: null handle");
    if (h->cfg.kind == SLB_KIND_MSCKF)
        return set_error(SLB_ERR_INVALID, "slb_set_nis_capture: UKF and USCKF batches only (the MSCKF update gates per feature and "
                                          "forms no whole-innovation distance)");
    if (on != 0 && on != 1) return set_error(SLB_ERR_INVALID, "slb_set_nis_capture: on must be 0 or 1");
    DeviceGuard guard(h->cfg.device);
    if (!on) {
        if (h->nis) SLB_CUDA(cudaFree(h->nis));   // (cudaFree waits for the kernels that still write it)
        h->nis = nullptr;
        return SLB_OK;
    }
    if (!h->nis) SLB_CUDA(cudaMalloc(&h->nis, (size_t)h->B * 8));
    SLB_CUDA(cudaMemset(h->nis, 0xff, (size_t)h->B * 8));   // all-ones bytes: a NaN in every entry
    return SLB_OK;
}
// doubles between consecutive instances' Q / R for a handle's noise layout (0 = shared)
static int q_stride(slb_handle h, int n) { return (h->noise & SLB_NOISE_Q_PER_INSTANCE) ? n * n : 0; }
static int r_stride(slb_handle h, int m) { return (h->noise & SLB_NOISE_R_PER_INSTANCE) ? m * m : 0; }
int slb_dof(slb_handle h) { return h ? h->L.N : SLB_ERR_INVALID; }
int slb_qdim(slb_handle h) { return h ? h->L.QD : SLB_ERR_INVALID; }

int slb_device_ptr(slb_handle h, int field, void **dev) {
    if (!h || !dev) return set_error(SLB_ERR_INVALID, "slb_device_ptr: null argument");
    switch (field) {
        case SLB_FIELD_MU: *dev = h->mu; return SLB_OK;
        case SLB_FIELD_P: *dev = h->P; return SLB_OK;
        case SLB_FIELD_STATUS: *dev = h->status; return SLB_OK;
        case SLB_FIELD_OUTLIERS: *dev = h->outliers; return SLB_OK;
        case SLB_FIELD_NIS:
            if (!h->nis) return set_error(SLB_ERR_INVALID, "slb_device_ptr: NIS capture is off (slb_set_nis_capture)");
            *dev = h->nis;
            return SLB_OK;
    }
    return set_error(SLB_ERR_INVALID, "slb_device_ptr: unknown field");
}

static int transfer(slb_handle h, int field, void *host, size_t count, cudaStream_t s, bool up) {
    if (!h || !host) return set_error(SLB_ERR_INVALID, "slb_upload/download: null argument");
    DeviceGuard guard(h->cfg.device);
    const slbd::BatchLayout &L = h->L;
    if (field == SLB_FIELD_STATUS || field == SLB_FIELD_OUTLIERS) {
        if (up) return set_error(SLB_ERR_INVALID, "slb_upload: status fields are read-only");
        if (count != (size_t)h->B) return set_error(SLB_ERR_INVALID, "slb_download: count must equal batch");
        SLB_CUDA(cudaMemcpyAsync(host, field == SLB_FIELD_STATUS ? h->status : h->outliers, (size_t)h->B * 4,
                                 cudaMemcpyDeviceToHost, s));
        SLB_CUDA(cudaStreamSynchronize(s));
        return SLB_OK;
    }
    if (field == SLB_FIELD_NIS) {
        if (up) return set_error(SLB_ERR_INVALID, "slb_upload: the NIS field is read-only");
        if (!h->nis) return set_error(SLB_ERR_INVALID, "slb_download: NIS capture is off (slb_set_nis_capture)");
        if (count != (size_t)h->B) return set_error(SLB_ERR_INVALID, "slb_download: count must equal batch");
        SLB_CUDA(cudaMemcpyAsync(host, h->nis, (size_t)h->B * 8, cudaMemcpyDeviceToHost, s));
        SLB_CUDA(cudaStreamSynchronize(s));
        return SLB_OK;
    }
    size_t per;
    if (field == SLB_FIELD_MU) per = L.QD;
    else if (field == SLB_FIELD_P) per = (size_t)L.N * L.N;
    else return set_error(SLB_ERR_INVALID, "slb_upload/download: unknown field");
    if (count == 0 || count % per != 0 || count > per * h->B)
        return set_error(SLB_ERR_INVALID, "slb_upload/download: count must be k * per-instance size, 1 <= k <= batch");
    const int nin = (int)(count / per);  // the first `nin` instances are transferred
    const int chunk = (int)(h->stage_bytes / (per * 8));
    double *hp = (double *)host;
    for (int b0 = 0; b0 < nin; b0 += chunk) {
        const int cnt = (nin - b0) < chunk ? (nin - b0) : chunk;
        const size_t bytes = (size_t)cnt * per * 8;
        const int64_t work = (int64_t)cnt * (field == SLB_FIELD_MU ? L.QD : up ? L.NP : L.N * L.N);
        const int tpb = 256;
        const int grid = (int)((work + tpb - 1) / tpb);
        if (up) {
            SLB_CUDA(cudaMemcpyAsync(h->stage, hp + (size_t)b0 * per, bytes, cudaMemcpyHostToDevice, s));
            if (field == SLB_FIELD_MU) mu_in<<<grid, tpb, 0, s>>>(h->stage, h->mu, L, b0, cnt);
            else P_in<<<grid, tpb, 0, s>>>(h->stage, h->P, L, b0, cnt);
            count_launch();
            SLB_CUDA(cudaGetLastError());
        } else {
            if (field == SLB_FIELD_MU) mu_out<<<grid, tpb, 0, s>>>(h->mu, h->stage, L, b0, cnt, 0, L.QD);
            else P_out<<<grid, tpb, 0, s>>>(h->P, h->stage, L, b0, cnt);
            count_launch();
            SLB_CUDA(cudaGetLastError());
            SLB_CUDA(cudaMemcpyAsync(hp + (size_t)b0 * per, h->stage, bytes, cudaMemcpyDeviceToHost, s));
        }
        // the staging buffer is reused by the next chunk (and by later calls)
        SLB_CUDA(cudaStreamSynchronize(s));
    }
    return SLB_OK;
}

int slb_upload(slb_handle h, int field, const void *host, size_t count, void *stream) {
    return transfer(h, field, const_cast<void *>(host), count, S(stream), true);
}
int slb_download(slb_handle h, int field, void *host, size_t count, void *stream) {
    return transfer(h, field, host, count, S(stream), false);
}

int slb_replicate(slb_handle h, int count, void *stream) {
    if (!h || count <= 0 || count > h->B) return set_error(SLB_ERR_INVALID, "slb_replicate: bad count");
    DeviceGuard guard(h->cfg.device);
    cudaStream_t s = S(stream);
    if (count == h->B) return SLB_OK;
    const int tpb = 256;
    int64_t w = (int64_t)h->L.QD * h->B;
    replicate<<<(unsigned)((w + tpb - 1) / tpb), tpb, 0, s>>>(h->mu, h->L, h->B, count, false);
    w = (int64_t)h->L.NP * h->B;
    replicate<<<(unsigned)((w + tpb - 1) / tpb), tpb, 0, s>>>(h->P, h->L, h->B, count, true);
    count_launch(2);
    SLB_CUDA(cudaGetLastError());
    return SLB_OK;
}

// ---- ukfom::ukf --------------------------------------------------------------------------------------
static int ukf_call(slb_handle h, int pm, int mm, bool pred, bool upd, const double *u, double dt, const double *Q,
                    const double *z, const double *R, int gate, void *stream) {
    if (!h || h->cfg.kind != SLB_KIND_UKF) return set_error(SLB_ERR_INVALID, "slb_ukf_*: handle is not a UKF batch");
    if (pred && (!u || !Q)) return set_error(SLB_ERR_INVALID, "slb_ukf_predict: u and Q are required");
    if (upd && (!z || !R)) return set_error(SLB_ERR_INVALID, "slb_ukf_update: z and R are required");
    DeviceGuard guard(h->cfg.device);
    FilterArgs a = make_args(h);
    a.u = u; a.dt = dt; a.Q = Q; a.z = z; a.R = R; a.gate = gate; a.m = 3;
    a.qs = q_stride(h, h->L.N); a.rs = r_stride(h, 3);
    return launch_ukf(h->cfg.layout, pm, mm, pred, upd, a, S(stream));
}
int slb_ukf_predict(slb_handle h, int pm, const double *u, double dt, const double *Q, void *stream) {
    return ukf_call(h, pm, 0, true, false, u, dt, Q, nullptr, nullptr, 0, stream);
}
int slb_ukf_update(slb_handle h, int mm, const double *z, const double *R, int gate_dof, void *stream) {
    return ukf_call(h, 0, mm, false, true, nullptr, 0.0, nullptr, z, R, gate_dof, stream);
}
int slb_ukf_step(slb_handle h, int pm, int mm, const double *u, double dt, const double *Q, const double *z,
                 const double *R, int gate_dof, void *stream) {
    return ukf_call(h, pm, mm, true, true, u, dt, Q, z, R, gate_dof, stream);
}

// Shared host-buffer step: the batch is cut into chunks that travel on a small ring of internal streams, so
// the H2D copy of chunk c+1 (u, z), the kernels of chunk c and the D2H copy of the posterior means of chunk
// c-1 overlap (PCIe is full duplex).  Q, R and the model parameters are small shared inputs copied first on
// the caller's stream; the call returns after everything has completed.
struct HostStep {
    int pm, mm, nu, m, nq, nparams, gate;
    double dt;
    const double *u, *Q, *params, *z, *R;
    double *mu_out;
};

static int launch_chunk(slb_handle h, const HostStep &hs, int b0, int cnt, const double *du, const double *dz,
                        const double *dQ, const double *dp, const double *dR, cudaStream_t st) {
    FilterArgs a = make_args(h);
    a.mu += h->L.mu(b0, 0);
    a.P += h->L.P(b0, 0, 0);
    a.status += b0;
    a.outliers += b0;
    if (a.nis) a.nis += b0;
    a.B = cnt;
    a.u = du; a.dt = hs.dt; a.Q = dQ; a.z = dz; a.R = dR; a.params = dp; a.gate = hs.gate; a.m = hs.m;
    switch (h->cfg.kind) {
        case SLB_KIND_UKF: return launch_ukf(h->cfg.layout, hs.pm, hs.mm, true, true, a, st);
        case SLB_KIND_USCKF: return launch_usckf(hs.pm, hs.mm, true, true, a, st);
        default: {
            int rc = launch_msckf_predict(hs.pm, a, st);
            return rc != SLB_OK ? rc : launch_msckf_update(hs.mm, a, st);
        }
    }
}

// Enqueues one predict+update step with host buffers on `s` (and the chunk ring forked from it): no synchronisation.
static int step_host_enqueue(slb_handle h, const HostStep &hs, cudaStream_t s) {
    double *du = h->stage, *dz = du + (size_t)h->B * hs.nu, *dmu = dz + (size_t)h->B * hs.m;
    double *dQ = h->shared_small, *dp = dQ + hs.nq * hs.nq, *dR = dp + hs.nparams;
    h->qr_nq = h->qr_m = 0;   // shared_small is rewritten: the zero-copy path's Q | R cache no longer describes it
    SLB_CUDA(cudaMemcpyAsync(dQ, hs.Q, (size_t)hs.nq * hs.nq * 8, cudaMemcpyHostToDevice, s));
    if (hs.nparams) SLB_CUDA(cudaMemcpyAsync(dp, hs.params, (size_t)hs.nparams * 8, cudaMemcpyHostToDevice, s));
    SLB_CUDA(cudaMemcpyAsync(dR, hs.R, (size_t)hs.m * hs.m * 8, cudaMemcpyHostToDevice, s));
    SLB_CUDA(cudaEventRecord(h->ev_start, s));
    // chunks of >= 8192 instances (multiples of 32 so no warp straddles a chunk), at most 8
    // The UKF step is short (a 65 536-instance fleet is 4.6 waves of CTAs, ~30 us per wave) and its PCIe traffic takes
    // as long as the kernel: fine chunks pay a whole wave each, so three chunks overlap best (measured on B200: 1 / 2 /
    // 3 / 4 / 6 / 8 chunks -> 391 / 417 / 317 / 378 / 390 / 364 us per step).  The USCKF / MSCKF steps are kernel-bound:
    // more, smaller chunks hide the transfers better (2 / 4 / 8 chunks -> 4.1e7 / 4.5e7 / 5.3e7 steps/s).
    int nchunk = h->cfg.kind == SLB_KIND_UKF ? h->B / 20000 : h->B / 8192;
    const int cmax = h->cfg.kind == SLB_KIND_UKF ? 3 : 8;
    nchunk = nchunk < 1 ? 1 : nchunk > cmax ? cmax : nchunk;
    {
        static const int forced = [] { const char *e = getenv("SLB_HOST_CHUNKS"); return e ? atoi(e) : 0; }();
        if (forced > 0) nchunk = forced;
    }
    const int per = ((h->B + nchunk - 1) / nchunk + 31) / 32 * 32;
    int used = 0;
    for (int c = 0, b0 = 0; b0 < h->B; ++c, b0 += per) {
        const int cnt = h->B - b0 < per ? h->B - b0 : per;
        cudaStream_t st = h->xs[c % SLB_NXS];
        if (c < SLB_NXS) { SLB_CUDA(cudaStreamWaitEvent(st, h->ev_start, 0)); used = c + 1; }
        SLB_CUDA(cudaMemcpyAsync(du + (size_t)b0 * hs.nu, hs.u + (size_t)b0 * hs.nu, (size_t)cnt * hs.nu * 8, cudaMemcpyHostToDevice, st));
        SLB_CUDA(cudaMemcpyAsync(dz + (size_t)b0 * hs.m, hs.z + (size_t)b0 * hs.m, (size_t)cnt * hs.m * 8, cudaMemcpyHostToDevice, st));
        const int rc = launch_chunk(h, hs, b0, cnt, du + (size_t)b0 * hs.nu, dz + (size_t)b0 * hs.m, dQ, dp, dR, st);
        if (rc != SLB_OK) return rc;
        if (hs.mu_out) {
            const int OL = h->out_len, work = cnt * OL, tpb = 256;
            double *dst = dmu + (size_t)b0 * OL;
            mu_out<<<(work + tpb - 1) / tpb, tpb, 0, st>>>(h->mu, dst, h->L, b0, cnt, h->out_off, OL);
            count_launch();
            SLB_CUDA(cudaGetLastError());
            SLB_CUDA(cudaMemcpyAsync(hs.mu_out + (size_t)b0 * OL, dst, (size_t)cnt * OL * 8, cudaMemcpyDeviceToHost, st));
        }
    }
    for (int i = 0; i < used; ++i) {
        SLB_CUDA(cudaEventRecord(h->ev_done[i], h->xs[i]));
        SLB_CUDA(cudaStreamWaitEvent(s, h->ev_done[i], 0));
    }
    return SLB_OK;
}

static bool is_pinned(const void *p) {
    if (!p) return true;
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return at.type == cudaMemoryTypeHost;
}
// Device-side alias of a page-locked host buffer for the zero-copy paths.  For cudaHostRegister'ed memory on systems
// without canUseHostPointerForRegisteredMem the alias differs from the host address; nullptr = no usable alias (the
// caller falls back to the copy pipeline).
static void *dev_alias_v(const void *p) {
    if (!p) return nullptr;
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) {
        cudaGetLastError();
        return nullptr;
    }
    if (at.type == cudaMemoryTypeDevice || at.type == cudaMemoryTypeManaged) return const_cast<void *>(p);
    return at.type == cudaMemoryTypeHost ? at.devicePointer : nullptr;
}
static const double *dev_alias(const double *p) { return (const double *)dev_alias_v(p); }
static double *dev_alias_m(double *p) { return (double *)dev_alias_v(p); }

static int step_host(slb_handle h, const HostStep &hs, void *stream, bool wait = true) {
    if (!h || !hs.u || !hs.Q || !hs.z || !hs.R) return set_error(SLB_ERR_INVALID, "slb_*_step_host: null argument");
    DeviceGuard guard(h->cfg.device);
    cudaStream_t s = S(stream);
    const size_t ub = (size_t)h->B * hs.nu * 8, zb = (size_t)h->B * hs.m * 8, mub = (size_t)h->B * h->L.QD * 8;
    const size_t small = (size_t)(hs.nq * hs.nq + hs.m * hs.m + hs.nparams) * 8;
    if (ub + zb + mub > h->stage_bytes || small > 128 * 1024)
        return set_error(SLB_ERR_INVALID, "slb_*_step_host: batch / shared inputs too large for the staging buffers");
    // With page-locked host buffers the whole pipeline is captured once and replayed (pageable copies cannot be captured).
    const bool graphable = is_pinned(hs.u) && is_pinned(hs.z) && is_pinned(hs.Q) && is_pinned(hs.R) && is_pinned(hs.params) &&
                           is_pinned(hs.mu_out);
    if (!graphable) {
        const int rc = step_host_enqueue(h, hs, s);
        if (rc != SLB_OK) return rc;
        SLB_CUDA(cudaStreamSynchronize(s));
        return SLB_OK;
    }
    // UKF: zero-copy.  The step is as short as its PCIe transfers, so instead of staging copies the kernel reads u / z
    // from the mapped (page-locked, UVA) host buffers and writes the posterior means straight back: transfers overlap
    // compute warp by warp.  Only the small shared Q / R are copied.  (SLB_ZERO_COPY=0 selects the copy pipeline.)
    static const bool zero_copy = [] { const char *e = getenv("SLB_ZERO_COPY"); return !e || atoi(e) != 0; }();
    const double *zu = dev_alias(hs.u), *zz = dev_alias(hs.z);
    double *zmu = dev_alias_m(hs.mu_out);
    if (zero_copy && zu && zz && (zmu || !hs.mu_out) && (h->cfg.kind == SLB_KIND_UKF || h->cfg.kind == SLB_KIND_USCKF)) {
        double *dQ = h->shared_small, *dR = dQ + hs.nq * hs.nq;
        const size_t qb = (size_t)hs.nq * hs.nq * 8, rb = (size_t)hs.m * hs.m * 8;
        const bool cacheable = hs.nq <= 12 && hs.m <= 9;
        if (!(cacheable && h->qr_nq == hs.nq && h->qr_m == hs.m && memcmp(h->qr_cache, hs.Q, qb) == 0 &&
              memcmp(h->qr_cache + 144, hs.R, rb) == 0)) {
            // (stream order protects the kernels of earlier steps that still read the previous values)
            SLB_CUDA(cudaMemcpyAsync(dQ, hs.Q, qb, cudaMemcpyHostToDevice, s));
            SLB_CUDA(cudaMemcpyAsync(dR, hs.R, rb, cudaMemcpyHostToDevice, s));
            h->qr_nq = h->qr_m = 0;
            if (cacheable) {
                memcpy(h->qr_cache, hs.Q, qb);
                memcpy(h->qr_cache + 144, hs.R, rb);
                h->qr_nq = hs.nq;
                h->qr_m = hs.m;
            }
        }
        FilterArgs a = make_args(h);
        a.u = zu; a.dt = hs.dt; a.Q = dQ; a.z = zz; a.R = dR; a.gate = hs.gate; a.m = hs.m;
        a.mu_out = zmu;
        const int rc = h->cfg.kind == SLB_KIND_UKF ? launch_ukf(h->cfg.layout, hs.pm, hs.mm, true, true, a, s)
                                                   : launch_usckf(hs.pm, hs.mm, true, true, a, s);
        if (rc != SLB_OK) return rc;
        if (wait) SLB_CUDA(cudaStreamSynchronize(s));
        return SLB_OK;
    }
    const int ki[8] = {hs.pm, hs.mm, hs.nu, hs.m, hs.nq, hs.nparams, hs.gate, h->out_off * 4096 + h->out_len};
    // the NIS array is a key too: toggling slb_set_nis_capture re-captures, so no replay writes a freed array or skips it
    const void *kp[7] = {hs.u, hs.Q, hs.params, hs.z, hs.R, hs.mu_out, h->nis};
    bool same = h->step_exec != nullptr && h->step_key_dt == hs.dt;
    for (int i = 0; i < 8 && same; ++i) same = h->step_key_i[i] == ki[i];
    for (int i = 0; i < 7 && same; ++i) same = h->step_key_p[i] == kp[i];
    if (!same) {
        if (h->step_exec) { cudaGraphExecDestroy(h->step_exec); h->step_exec = nullptr; }
        const int64_t n0 = slb_launch_count();
        SLB_CUDA(cudaStreamBeginCapture(h->cap_stream, cudaStreamCaptureModeThreadLocal));
        const int rc = step_host_enqueue(h, hs, h->cap_stream);
        cudaGraph_t g = nullptr;
        const cudaError_t ce = cudaStreamEndCapture(h->cap_stream, &g);
        const int nk = (int)(slb_launch_count() - n0);
        count_launch(-nk);  // captured, not executed
        if (rc != SLB_OK || ce != cudaSuccess || !g) {
            if (g) cudaGraphDestroy(g);
            cudaGetLastError();
            return rc != SLB_OK ? rc : set_error(SLB_ERR_CUDA, "slb_*_step_host: stream capture failed", ce);
        }
        const cudaError_t ie = cudaGraphInstantiate(&h->step_exec, g, 0);
        cudaGraphDestroy(g);
        if (ie != cudaSuccess) {
            h->step_exec = nullptr;
            return set_error(SLB_ERR_CUDA, "slb_*_step_host: cudaGraphInstantiate", ie);
        }
        h->step_kernels = nk;
        h->step_key_dt = hs.dt;
        for (int i = 0; i < 8; ++i) h->step_key_i[i] = ki[i];
        for (int i = 0; i < 7; ++i) h->step_key_p[i] = kp[i];
    }
    SLB_CUDA(cudaGraphLaunch(h->step_exec, s));
    count_launch(h->step_kernels);
    if (wait) SLB_CUDA(cudaStreamSynchronize(s));
    return SLB_OK;
}
static int ukf_step_host(slb_handle h, int pm, int mm, const double *u_host, double dt, const double *Q_host,
                         const double *z_host, const double *R_host, int gate_dof, double *mu_out_host, void *stream, bool wait) {
    if (!h || h->cfg.kind != SLB_KIND_UKF) return set_error(SLB_ERR_INVALID, "slb_ukf_step_host: handle is not a UKF batch");
    if (h->noise) return set_error(SLB_ERR_INVALID, "slb_ukf_step_host: per-instance noise (slb_set_noise_layout) is device-resident only");
    if (mm != SLB_MM_GPS_POS) return set_error(SLB_ERR_INVALID, "ukf: unsupported measurement model");
    const HostStep hs = {pm, mm, pm_nu(pm), 3, h->L.N, 0, gate_dof, dt, u_host, Q_host, nullptr, z_host, R_host, mu_out_host};
    return step_host(h, hs, stream, wait);
}
int slb_ukf_step_host(slb_handle h, int pm, int mm, const double *u_host, double dt, const double *Q_host,
                      const double *z_host, const double *R_host, int gate_dof, double *mu_out_host, void *stream) {
    return ukf_step_host(h, pm, mm, u_host, dt, Q_host, z_host, R_host, gate_dof, mu_out_host, stream, true);
}
int slb_ukf_step_host_async(slb_handle h, int pm, int mm, const double *u_host, double dt, const double *Q_host,
                            const double *z_host, const double *R_host, int gate_dof, double *mu_out_host, void *stream) {
    return ukf_step_host(h, pm, mm, u_host, dt, Q_host, z_host, R_host, gate_dof, mu_out_host, stream, false);
}
// Completes every step enqueued on `stream` by the *_step_host_async entry points (the host buffers passed to them
// may be reused / read afterwards).
int slb_wait(slb_handle h, void *stream) {
    if (!h) return set_error(SLB_ERR_INVALID, "slb_wait: null argument");
    DeviceGuard guard(h->cfg.device);
    SLB_CUDA(cudaStreamSynchronize(S(stream)));
    return SLB_OK;
}

// ---- localization::Usckf -----------------------------------------------------------------------------
static int usckf_call(slb_handle h, int pm, int mm, bool pred, bool upd, const double *u, double dt, const double *Q,
                      const double *z, const double *R, int gate, void *stream) {
    if (!h || h->cfg.kind != SLB_KIND_USCKF) return set_error(SLB_ERR_INVALID, "slb_usckf_*: handle is not a USCKF batch");
    if (pred && (!u || !Q)) return set_error(SLB_ERR_INVALID, "slb_usckf_predict: u and Q are required");
    if (upd && (!z || !R)) return set_error(SLB_ERR_INVALID, "slb_usckf_update: z and R are required");
    DeviceGuard guard(h->cfg.device);
    FilterArgs a = make_args(h);
    a.u = u; a.dt = dt; a.Q = Q; a.z = z; a.R = R; a.gate = gate; a.m = h->cfg.nk;
    a.qs = q_stride(h, 12); a.rs = r_stride(h, h->cfg.nk);
    return launch_usckf(pm, mm, pred, upd, a, S(stream));
}
int slb_usckf_predict(slb_handle h, int pm, const double *u, double dt, const double *Q, void *stream) {
    return usckf_call(h, pm, 0, true, false, u, dt, Q, nullptr, nullptr, 0, stream);
}
int slb_usckf_update(slb_handle h, int mm, const double *z, const double *R, int gate_dof, void *stream) {
    return usckf_call(h, 0, mm, false, true, nullptr, 0.0, nullptr, z, R, gate_dof, stream);
}
int slb_usckf_step(slb_handle h, int pm, int mm, const double *u, double dt, const double *Q, const double *z,
                   const double *R, int gate_dof, void *stream) {
    return usckf_call(h, pm, mm, true, true, u, dt, Q, z, R, gate_dof, stream);
}
static int usckf_step_host(slb_handle h, int pm, int mm, const double *u_host, double dt, const double *Q_host,
                           const double *z_host, const double *R_host, int gate_dof, double *mu_out_host, void *stream, bool wait) {
    if (!h || h->cfg.kind != SLB_KIND_USCKF) return set_error(SLB_ERR_INVALID, "slb_usckf_step_host: handle is not a USCKF batch");
    if (h->noise) return set_error(SLB_ERR_INVALID, "slb_usckf_step_host: per-instance noise (slb_set_noise_layout) is device-resident only");
    const HostStep hs = {pm, mm, pm_nu(pm), h->cfg.nk, 12, 0, gate_dof, dt, u_host, Q_host, nullptr, z_host, R_host, mu_out_host};
    return step_host(h, hs, stream, wait);
}
int slb_usckf_step_host(slb_handle h, int pm, int mm, const double *u_host, double dt, const double *Q_host,
                        const double *z_host, const double *R_host, int gate_dof, double *mu_out_host, void *stream) {
    return usckf_step_host(h, pm, mm, u_host, dt, Q_host, z_host, R_host, gate_dof, mu_out_host, stream, true);
}
int slb_usckf_step_host_async(slb_handle h, int pm, int mm, const double *u_host, double dt, const double *Q_host,
                              const double *z_host, const double *R_host, int gate_dof, double *mu_out_host, void *stream) {
    return usckf_step_host(h, pm, mm, u_host, dt, Q_host, z_host, R_host, gate_dof, mu_out_host, stream, false);
}
int slb_usckf_clone(slb_handle h, int mode, void *stream) {
    if (!h || h->cfg.kind != SLB_KIND_USCKF) return set_error(SLB_ERR_INVALID, "slb_usckf_clone: handle is not a USCKF batch");
    DeviceGuard guard(h->cfg.device);
    FilterArgs a = make_args(h);
    return launch_usckf_clone(mode, a, S(stream));
}
int slb_usckf_set_measurement(slb_handle h, int mode, const double *z, const double *R, void *stream) {
    if (!h || h->cfg.kind != SLB_KIND_USCKF) return set_error(SLB_ERR_INVALID, "slb_usckf_set_measurement: handle is not a USCKF batch");
    if (!z || !R) return set_error(SLB_ERR_INVALID, "slb_usckf_set_measurement: z and R are required");
    DeviceGuard guard(h->cfg.device);
    FilterArgs a = make_args(h);
    a.z = z; a.R = R;
    a.rs = r_stride(h, mode == SLB_STATEK ? h->cfg.nk : h->cfg.nl);
    return launch_usckf_set_measurement(mode, a, S(stream));
}

// ---- localization::Msckf -----------------------------------------------------------------------------
int slb_msckf_predict(slb_handle h, int pm, const double *u, double dt, const double *Q, void *stream) {
    if (!h || h->cfg.kind != SLB_KIND_MSCKF) return set_error(SLB_ERR_INVALID, "slb_msckf_predict: handle is not an MSCKF batch");
    if (!u || !Q) return set_error(SLB_ERR_INVALID, "slb_msckf_predict: u and Q are required");
    DeviceGuard guard(h->cfg.device);
    FilterArgs a = make_args(h);
    a.u = u; a.dt = dt; a.Q = Q;
    a.qs = q_stride(h, 12);
    return launch_msckf_predict(pm, a, S(stream));
}
int slb_msckf_update(slb_handle h, int mm, const double *params, int m, const double *z, const double *R, int gate,
                     void *stream) {
    if (!h || h->cfg.kind != SLB_KIND_MSCKF) return set_error(SLB_ERR_INVALID, "slb_msckf_update: handle is not an MSCKF batch");
    if (!params || !z || !R || m <= 0 || (m & 1)) return set_error(SLB_ERR_INVALID, "slb_msckf_update: bad arguments");
    DeviceGuard guard(h->cfg.device);
    FilterArgs a = make_args(h);
    a.params = params; a.m = m; a.z = z; a.R = R; a.gate = gate;
    return launch_msckf_update(mm, a, S(stream));
}

int slb_msckf_update_ekf(slb_handle h, int mm, const double *params, int m, const double *z, const double *R, int gate,
                         void *stream) {
    if (!h || h->cfg.kind != SLB_KIND_MSCKF) return set_error(SLB_ERR_INVALID, "slb_msckf_update_ekf: handle is not an MSCKF batch");
    if (!params || !z || !R || m <= 0 || (m & 1)) return set_error(SLB_ERR_INVALID, "slb_msckf_update_ekf: bad arguments");
    DeviceGuard guard(h->cfg.device);
    FilterArgs a = make_args(h);
    a.params = params; a.m = m; a.z = z; a.R = R; a.gate = gate;
    return launch_msckf_update_ekf(mm, a, S(stream));
}

// predict + update with HOST buffers (the end-to-end arm of bench.py): u | z staged on the device, the
// posterior means copied back.  Q, R and the landmark parameters are small shared inputs.
static int msckf_step_host(slb_handle h, int pm, int mm, const double *u_host, double dt, const double *Q_host,
                           const double *params_host, int nparams, int m, const double *z_host, const double *R_host,
                           int gate, double *mu_out_host, void *stream, bool wait);
int slb_msckf_step_host(slb_handle h, int pm, int mm, const double *u_host, double dt, const double *Q_host,
                        const double *params_host, int nparams, int m, const double *z_host, const double *R_host,
                        int gate, double *mu_out_host, void *stream) {
    return msckf_step_host(h, pm, mm, u_host, dt, Q_host, params_host, nparams, m, z_host, R_host, gate, mu_out_host, stream, true);
}
int slb_msckf_step_host_async(slb_handle h, int pm, int mm, const double *u_host, double dt, const double *Q_host,
                              const double *params_host, int nparams, int m, const double *z_host, const double *R_host,
                              int gate, double *mu_out_host, void *stream) {
    return msckf_step_host(h, pm, mm, u_host, dt, Q_host, params_host, nparams, m, z_host, R_host, gate, mu_out_host, stream, false);
}
static int msckf_step_host(slb_handle h, int pm, int mm, const double *u_host, double dt, const double *Q_host,
                           const double *params_host, int nparams, int m, const double *z_host, const double *R_host,
                           int gate, double *mu_out_host, void *stream, bool wait) {
    if (!h || h->cfg.kind != SLB_KIND_MSCKF) return set_error(SLB_ERR_INVALID, "slb_msckf_step_host: handle is not an MSCKF batch");
    if (h->noise) return set_error(SLB_ERR_INVALID, "slb_msckf_step_host: per-instance noise (slb_set_noise_layout) is device-resident only");
    if (!u_host || !Q_host || !params_host || !z_host || !R_host || m <= 0 || nparams <= 0)
        return set_error(SLB_ERR_INVALID, "slb_msckf_step_host: null argument");
    const HostStep hs = {pm, mm, pm_nu(pm), m, 12, nparams, gate, dt, u_host, Q_host, params_host, z_host, R_host, mu_out_host};
    if (mm != SLB_MM_MSCKF_REPROJ || (m & 1)) return set_error(SLB_ERR_INVALID, "slb_msckf_step_host: bad measurement model / m");
    return step_host(h, hs, stream, wait);
}

// ---- localization::DataModel -------------------------------------------------------------------------
int slb_datamodel_fuse(int d, int64_t n, const double *x1, const double *C1, const double *x2, const double *C2,
                       double *xo, double *Co, void *stream) {
    if (!x1 || !C1 || !x2 || !C2 || !xo || !Co || n < 0) return set_error(SLB_ERR_INVALID, "slb_datamodel_fuse: bad arguments");
    return launch_fusion(d, n, 0, x1, C1, x2, C2, xo, Co, S(stream));
}
int slb_datamodel_addsub(int d, int64_t n, int sign, const double *x1, const double *C1, const double *x2,
                         const double *C2, double *xo, double *Co, void *stream) {
    if (!x1 || !C1 || !x2 || !C2 || !xo || !Co || n < 0 || sign == 0) return set_error(SLB_ERR_INVALID, "slb_datamodel_addsub: bad arguments");
    return launch_fusion(d, n, sign > 0 ? 1 : -1, x1, C1, x2, C2, xo, Co, S(stream));
}
int slb_datamodel_fuse_host(int d, int64_t n, const double *x1, const double *C1, const double *x2, const double *C2,
                            double *xo, double *Co) {
    if (!x1 || !C1 || !x2 || !C2 || !xo || !Co || n < 0) return set_error(SLB_ERR_INVALID, "slb_datamodel_fuse_host: bad arguments");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        return set_error(SLB_ERR_NO_DEVICE, "slb_datamodel_fuse_host: no CUDA device (no CPU fallback)");
    }
    if (n == 0) return SLB_OK;
    // Page-locked buffers: zero-copy.  The kernel stages its covariance tiles with coalesced LDGSTS and writes its
    // results with coalesced stores, which work just as well against mapped host memory: the 1 GB of H2D / D2H
    // traffic of a 1M-pair step overlaps in both directions and with the arithmetic, and nothing is allocated.
    {
        static const bool zero_copy = [] { const char *e = getenv("SLB_ZERO_COPY"); return !e || atoi(e) != 0; }();
        const double *a1 = dev_alias(x1), *A1 = dev_alias(C1), *a2 = dev_alias(x2), *A2 = dev_alias(C2);
        double *ao = dev_alias_m(xo), *Ao = dev_alias_m(Co);
        if (zero_copy && is_pinned(x1) && is_pinned(C1) && is_pinned(x2) && is_pinned(C2) && is_pinned(xo) && is_pinned(Co) &&
            a1 && A1 && a2 && A2 && ao && Ao) {
            const int rc = launch_fusion(d, n, 0, a1, A1, a2, A2, ao, Ao, 0);
            if (rc != SLB_OK) return rc;
            SLB_CUDA(cudaStreamSynchronize(0));
            return SLB_OK;
        }
    }
    const size_t xb = (size_t)n * d * 8, cb = (size_t)n * d * d * 8;
    double *buf = nullptr;
    SLB_CUDA(cudaMalloc(&buf, 2 * xb + 2 * cb));
    double *dx1 = buf, *dx2 = dx1 + (size_t)n * d, *dC1 = dx2 + (size_t)n * d, *dC2 = dC1 + (size_t)n * d * d;
    cudaError_t e = cudaMemcpyAsync(dx1, x1, xb, cudaMemcpyHostToDevice, 0);
    if (e == cudaSuccess) e = cudaMemcpyAsync(dx2, x2, xb, cudaMemcpyHostToDevice, 0);
    if (e == cudaSuccess) e = cudaMemcpyAsync(dC1, C1, cb, cudaMemcpyHostToDevice, 0);
    if (e == cudaSuccess) e = cudaMemcpyAsync(dC2, C2, cb, cudaMemcpyHostToDevice, 0);
    int rc = SLB_OK;
    if (e == cudaSuccess) rc = launch_fusion(d, n, 0, dx1, dC1, dx2, dC2, dx1, dC1, 0);
    if (e == cudaSuccess && rc == SLB_OK) e = cudaMemcpyAsync(xo, dx1, xb, cudaMemcpyDeviceToHost, 0);
    if (e == cudaSuccess && rc == SLB_OK) e = cudaMemcpyAsync(Co, dC1, cb, cudaMemcpyDeviceToHost, 0);
    if (e == cudaSuccess) e = cudaStreamSynchronize(0);
    cudaFree(buf);
    if (e != cudaSuccess) return set_error(SLB_ERR_CUDA, "slb_datamodel_fuse_host", e);
    return rc;
}

// ---- device buffers ----------------------------------------------------------------------------------
int slb_dev_alloc(size_t bytes, void **dev) {
    if (!dev) return set_error(SLB_ERR_INVALID, "slb_dev_alloc: null argument");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        return set_error(SLB_ERR_NO_DEVICE, "slb_dev_alloc: no CUDA device (this engine has no CPU fallback)");
    }
    SLB_CUDA(cudaMalloc(dev, bytes ? bytes : 8));
    return SLB_OK;
}
int slb_dev_free(void *dev) {
    if (dev) SLB_CUDA(cudaFree(dev));
    return SLB_OK;
}
int slb_dev_copy(void *dst, const void *src, size_t bytes, int kind, void *stream) {
    if (!dst || !src) return set_error(SLB_ERR_INVALID, "slb_dev_copy: null argument");
    const cudaMemcpyKind k = kind == 1 ? cudaMemcpyHostToDevice : kind == 2 ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice;
    SLB_CUDA(cudaMemcpyAsync(dst, src, bytes, k, S(stream)));
    if (kind == 2) SLB_CUDA(cudaStreamSynchronize(S(stream)));
    return SLB_OK;
}

// ---- diagnostics -------------------------------------------------------------------------------------
int slb_status_ex(slb_handle h, int64_t *counts, int nbits, void *stream) {
    if (!h || !counts || nbits < 1 || nbits > SLB_NSTATUS) return set_error(SLB_ERR_INVALID, "slb_status: bad argument");
    DeviceGuard guard(h->cfg.device);
    cudaStream_t s = S(stream);
    SLB_CUDA(cudaMemsetAsync(h->counts_dev, 0, 8 * sizeof(int64_t), s));
    int grid = (h->B + 255) / 256;
    if (grid > 1184) grid = 1184;
    status_count<<<grid, 256, 0, s>>>(h->status, h->B, (unsigned long long *)h->counts_dev);
    count_launch();
    SLB_CUDA(cudaGetLastError());
    SLB_CUDA(cudaMemcpyAsync(counts, h->counts_dev, (size_t)nbits * sizeof(int64_t), cudaMemcpyDeviceToHost, s));
    SLB_CUDA(cudaStreamSynchronize(s));
    return SLB_OK;
}
int slb_status(slb_handle h, int64_t counts[4], void *stream) { return slb_status_ex(h, counts, 4, stream); }
int slb_clear_status(slb_handle h, void *stream) {
    if (!h) return set_error(SLB_ERR_INVALID, "slb_clear_status: null argument");
    DeviceGuard guard(h->cfg.device);
    SLB_CUDA(cudaMemsetAsync(h->status, 0, (size_t)h->B * 4, S(stream)));
    SLB_CUDA(cudaMemsetAsync(h->outliers, 0, (size_t)h->B * 4, S(stream)));
    return SLB_OK;
}
int slb_bench_fp64_peak(double *tflops_out) {
    if (!tflops_out) return set_error(SLB_ERR_INVALID, "slb_bench_fp64_peak: null argument");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        return set_error(SLB_ERR_NO_DEVICE, "slb_bench_fp64_peak: no CUDA device");
    }
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    double *sink = nullptr;
    SLB_CUDA(cudaMalloc(&sink, 8));
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0);
    cudaEventCreate(&e1);
    const int iters = 4096, grid = sms * 8;
    double best = 0.0;
    for (int rep = 0; rep < 5; ++rep) {
        cudaEventRecord(e0, 0);
        fp64_peak_kernel<<<grid, 256, 0, 0>>>(sink, iters, 1.0000001, 0.9999999);
        cudaEventRecord(e1, 0);
        cudaEventSynchronize(e1);
        float ms = 0;
        cudaEventElapsedTime(&ms, e0, e1);
        const double fl = 2.0 * 16 * (double)iters * 256 * grid;
        const double tf = fl / (ms * 1e-3) * 1e-12;
        if (rep > 0 && tf > best) best = tf;
    }
    count_launch(5);
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    cudaFree(sink);
    SLB_CUDA(cudaGetLastError());
    *tflops_out = best;
    return SLB_OK;
}

int slb_ensemble_stats(slb_handle h, double *out_dev, void *stream) {
    if (!h || !out_dev) return set_error(SLB_ERR_INVALID, "slb_ensemble_stats: null argument");
    DeviceGuard guard(h->cfg.device);
    cudaStream_t s = S(stream);
    const int N = h->L.N;
    if (N * N + N > STAT_TPB * STAT_MAXACC) return set_error(SLB_ERR_INVALID, "slb_ensemble_stats: state too large");
    SLB_CUDA(cudaMemsetAsync(out_dev, 0, (size_t)(1 + N + N * N) * 8, s));
    const int nchunks = (h->B + STAT_CHUNK - 1) / STAT_CHUNK;
    const int grid = nchunks < 296 ? nchunks : 296;
    ensemble_stats_kernel<<<grid, STAT_TPB, (size_t)STAT_CHUNK * N * 8, s>>>(h->mu, h->B, h->L, out_dev);
    count_launch();
    SLB_CUDA(cudaGetLastError());
    return SLB_OK;
}

// ---- filter consistency: NEES against a per-instance truth, NIS of the last update --------------------------------
// t0 and t0 + n must not cut a 3-DOF block; n = 0 (with no truth) asks for the NIS sums only
static bool consistency_range_ok(const slbd::BatchLayout &L, const double *truth, int t0, int n) {
    if (!truth) return n == 0 && t0 == 0;
    const int nb3 = 3 * L.nblk;
    if (n <= 0 || t0 < 0 || t0 + n > L.N) return false;
    if (t0 < nb3 && t0 % 3 != 0) return false;
    if (t0 + n < nb3 && (t0 + n) % 3 != 0) return false;
    return true;
}
int slb_consistency_stats(slb_handle h, const double *truth_dev, int t0, int n, double *nees_dev, double *out_dev,
                          void *stream) {
    if (!h || !out_dev) return set_error(SLB_ERR_INVALID, "slb_consistency_stats: null argument");
    if (!consistency_range_ok(h->L, truth_dev, t0, n))
        return set_error(SLB_ERR_INVALID, "slb_consistency_stats: [t0, t0 + n) must be a non-empty range of the tangent "
                                          "coordinates that cuts no 3-DOF block (n = 0 and t0 = 0 without a truth)");
    DeviceGuard guard(h->cfg.device);
    cudaStream_t s = S(stream);
    SLB_CUDA(cudaMemsetAsync(out_dev, 0, 6 * sizeof(double), s));
    return launch_consistency(h, truth_dev, t0, n, nees_dev, out_dev, s);
}

// ---- checkSigmaPoints() -----------------------------------------------------------------------------------
int slb_check_sigma_points(slb_handle h, int32_t *flags_dev, double *diff_dev, void *stream) {
    if (!h || !flags_dev) return set_error(SLB_ERR_INVALID, "slb_check_sigma_points: null argument");
    if (h->cfg.kind == SLB_KIND_UKF)
        return set_error(SLB_ERR_INVALID, "slb_check_sigma_points: Usckf / Msckf batches only (the reference's ukfom::ukf has no checkSigmaPoints)");
    DeviceGuard guard(h->cfg.device);
    return launch_check_sigma_points(h, flags_dev, diff_dev, S(stream));
}

// ---- multi-GPU: ensemble statistics merged over an NCCL communicator ------------------------------------------
// NCCL is resolved at run time (dlopen of libnccl.so.2: the copy the process already carries, e.g. torch's, or the
// system one), so libslb.so has no link-time dependency on it and loads on machines without NCCL.
namespace {
struct NcclApi {
    void *lib = nullptr;
    ncclResult_t (*GetUniqueId)(ncclUniqueId *) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t *, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*AllReduce)(const void *, void *, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
    const char *(*GetErrorString)(ncclResult_t) = nullptr;
    bool ok = false;
};
NcclApi &nccl_api() {
    static NcclApi a = [] {
        NcclApi x;
        x.lib = dlopen("libnccl.so.2", RTLD_NOW | RTLD_LOCAL);
        if (!x.lib) x.lib = dlopen("libnccl.so", RTLD_NOW | RTLD_LOCAL);
        if (!x.lib) return x;
        x.GetUniqueId = (decltype(x.GetUniqueId))dlsym(x.lib, "ncclGetUniqueId");
        x.CommInitRank = (decltype(x.CommInitRank))dlsym(x.lib, "ncclCommInitRank");
        x.CommDestroy = (decltype(x.CommDestroy))dlsym(x.lib, "ncclCommDestroy");
        x.AllReduce = (decltype(x.AllReduce))dlsym(x.lib, "ncclAllReduce");
        x.GetErrorString = (decltype(x.GetErrorString))dlsym(x.lib, "ncclGetErrorString");
        x.ok = x.GetUniqueId && x.CommInitRank && x.CommDestroy && x.AllReduce;
        return x;
    }();
    return a;
}
int nccl_fail(const char *what, ncclResult_t r) {
    NcclApi &a = nccl_api();
    char buf[256];
    snprintf(buf, sizeof(buf), "%s: %s", what, a.GetErrorString ? a.GetErrorString(r) : "NCCL error");
    return set_error(SLB_ERR_NCCL, buf);
}
}  // namespace

int slb_nccl_unique_id(void *id128) {
    if (!id128) return set_error(SLB_ERR_INVALID, "slb_nccl_unique_id: null argument");
    NcclApi &a = nccl_api();
    if (!a.ok) return set_error(SLB_ERR_NCCL, "NCCL is not available (dlopen libnccl.so.2 failed)");
    static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId is 128 bytes");
    const ncclResult_t r = a.GetUniqueId((ncclUniqueId *)id128);
    return r == ncclSuccess ? SLB_OK : nccl_fail("ncclGetUniqueId", r);
}
int slb_nccl_comm_init(void **comm, int nranks, const void *id128, int rank, int device) {
    if (!comm || !id128 || nranks < 1 || rank < 0 || rank >= nranks) return set_error(SLB_ERR_INVALID, "slb_nccl_comm_init: bad argument");
    NcclApi &a = nccl_api();
    if (!a.ok) return set_error(SLB_ERR_NCCL, "NCCL is not available (dlopen libnccl.so.2 failed)");
    DeviceGuard guard(device);
    ncclUniqueId id;
    memcpy(&id, id128, sizeof(id));
    ncclComm_t c = nullptr;
    const ncclResult_t r = a.CommInitRank(&c, nranks, id, rank);
    if (r != ncclSuccess) return nccl_fail("ncclCommInitRank", r);
    *comm = c;
    return SLB_OK;
}
int slb_nccl_comm_destroy(void *comm) {
    if (!comm) return SLB_OK;
    NcclApi &a = nccl_api();
    if (!a.ok) return set_error(SLB_ERR_NCCL, "NCCL is not available");
    const ncclResult_t r = a.CommDestroy((ncclComm_t)comm);
    return r == ncclSuccess ? SLB_OK : nccl_fail("ncclCommDestroy", r);
}
int slb_gather_stats(slb_handle h, void *nccl_comm, double *out_dev, void *stream) {
    if (!h || !out_dev) return set_error(SLB_ERR_INVALID, "slb_gather_stats: null argument");
    const int rc = slb_ensemble_stats(h, out_dev, stream);
    if (rc != SLB_OK || !nccl_comm) return rc;   // no communicator: this device's shard only
    NcclApi &a = nccl_api();
    if (!a.ok) return set_error(SLB_ERR_NCCL, "NCCL is not available (dlopen libnccl.so.2 failed)");
    DeviceGuard guard(h->cfg.device);
    const size_t n = (size_t)1 + h->L.N + (size_t)h->L.N * h->L.N;
    const ncclResult_t r = a.AllReduce(out_dev, out_dev, n, ncclDouble, ncclSum, (ncclComm_t)nccl_comm, S(stream));
    return r == ncclSuccess ? SLB_OK : nccl_fail("ncclAllReduce", r);
}
int slb_gather_consistency(slb_handle h, void *nccl_comm, const double *truth_dev, int t0, int n, double *nees_dev,
                           double *out_dev, void *stream) {
    if (!h || !out_dev) return set_error(SLB_ERR_INVALID, "slb_gather_consistency: null argument");
    const int rc = slb_consistency_stats(h, truth_dev, t0, n, nees_dev, out_dev, stream);
    if (rc != SLB_OK || !nccl_comm) return rc;   // no communicator: this device's shard only
    NcclApi &a = nccl_api();
    if (!a.ok) return set_error(SLB_ERR_NCCL, "NCCL is not available (dlopen libnccl.so.2 failed)");
    DeviceGuard guard(h->cfg.device);
    const ncclResult_t r = a.AllReduce(out_dev, out_dev, 6, ncclDouble, ncclSum, (ncclComm_t)nccl_comm, S(stream));
    return r == ncclSuccess ? SLB_OK : nccl_fail("ncclAllReduce", r);
}

}  // extern "C"
