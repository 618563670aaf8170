// slb_internal.h -- shared declarations between the translation units of libslb.so.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/slb.h"
#include "slb_math.cuh"

constexpr int SLB_NXS = 3;  // internal streams of the *_step_host pipelines

// The (featuresk, featuresk_l) sizes the USCKF update is instantiated for.  The reference's feature vectors are dynamic
// (State.hpp:539-540, setMeasurement resizes Pk, Usckf.hpp:346-348); a batch has fixed sizes chosen at slb_create,
// which rejects what is not in this list.  N = 36 + nk + nl <= 48 keeps the accumulator tiles in registers.
#define SLB_USCKF_SHAPES(X) X(3, 0) X(3, 3) X(3, 6) X(3, 9) X(6, 0) X(6, 3) X(6, 6) X(9, 0) X(9, 3)

struct slb_batch_s {
    slb_config cfg;
    int B;        // instances
    slbd::BatchLayout L;  // dimensions and storage of mu and P
    double *mu;   // L.mu_size(B) doubles
    double *P;    // L.P_size(B) doubles
    int32_t *status;
    int32_t *outliers;
    // staging for the *_host entry points and upload/download
    double *stage;        // device scratch, stage_bytes long
    size_t stage_bytes;
    double *shared_small; // device copy of Q / R / params passed from host pointers
    int64_t *counts_dev;  // 4 counters for slb_status
    int32_t *misc_dev;    // 16 ints of per-launch scratch flags (e.g. "R is diagonal" for the MSCKF EKF update)
    cudaStream_t xs[SLB_NXS];  // chunk ring of the *_step_host entry points
    // the *_step_host pipeline captured as a CUDA graph (replayed while the caller keeps passing the same pinned
    // buffers and parameters: one cudaGraphLaunch instead of ~30 stream calls per step)
    cudaStream_t cap_stream;
    cudaGraphExec_t step_exec;
    int step_kernels;          // kernel launches inside the captured step
    int step_key_i[8];
    double step_key_dt;
    const void *step_key_p[7];   // the host buffers, and the NIS array the captured kernels write (slb_set_nis_capture)
    cudaEvent_t ev_start, ev_done[SLB_NXS];
    int out_off, out_len;      // slb_set_output_slice: part of the q-vector the *_step_host entry points copy back
    int noise;                 // slb_set_noise_layout: SLB_NOISE_* flags (0 = Q and R shared by the batch)
    double *nis;               // slb_set_nis_capture: B doubles, the m2 of every instance's last update (nullptr = off)
    // zero-copy *_step_host: host copy of the Q | R last uploaded to shared_small (the upload is skipped while the caller
    // keeps passing the same values: two tiny DMA operations per step are 10 % of a UKFoM step)
    double qr_cache[144 + 81];
    int qr_nq, qr_m;           // 0 = nothing cached
};

namespace slb {

int set_error(int code, const char *what, cudaError_t ce = cudaSuccess);
void count_launch(int n = 1);

#define SLB_CUDA(call)                                                        \
    do {                                                                      \
        cudaError_t e_ = (call);                                              \
        if (e_ != cudaSuccess) return slb::set_error(SLB_ERR_CUDA, #call, e_); \
    } while (0)

// Every entry point that takes a handle runs on the handle's device and leaves the caller's current device as it
// found it (several handles on several devices may be driven from one thread).
struct DeviceGuard {
    int prev = -1;
    bool switched = false;
    explicit DeviceGuard(int dev) {
        if (cudaGetDevice(&prev) == cudaSuccess && prev != dev) switched = cudaSetDevice(dev) == cudaSuccess;
    }
    ~DeviceGuard() {
        if (switched) cudaSetDevice(prev);
    }
    DeviceGuard(const DeviceGuard &) = delete;
    DeviceGuard &operator=(const DeviceGuard &) = delete;
};

struct FilterArgs {
    double *mu;
    double *P;
    int32_t *status;
    int32_t *outliers;
    int B;
    int stride, pstride, qstride;
    const double *u;
    double dt;
    const double *Q;
    const double *z;
    const double *R;
    const double *params;
    int m;
    int gate;
    int nk, nl, k;
    // per-instance noise (slb_set_noise_layout): qs / rs = doubles between consecutive instances' Q / R, 0 = one matrix
    // shared by the batch; the launchers select the kernels' per-instance instantiations when one of them is set.  The
    // two fill alignment holes: the kernels' parameter layout (size, every other member's offset) is as without them.
    int qs;
    int32_t *misc;
    int prefetch;     // USCKF step: L2-prefetch the record of instance (i + prefetch); 0 = off
    int rs;
    double *mu_out;   // optional instance-major copy of the posterior means (may be mapped host memory), B x out_len
    int out_off, out_len;  // the slice [out_off, out_off + out_len) of the q-vector that goes to mu_out
    // NIS capture (slb_set_nis_capture): the UKF / USCKF update writes the m2 its gate was given to nis[inst] (NaN when
    // the update stopped before forming it); the launchers select the kernels' NIS instantiations when it is set.  The
    // last member, so every other one keeps its offset and the kernels without NIS compile as before.
    double *nis;
};
static_assert(sizeof(FilterArgs) == 160, "FilterArgs layout");

// slb_ukf.cu
int launch_ukf(int layout, int pm, int mm, bool predict, bool update, const FilterArgs &a, cudaStream_t s);
// slb_usckf.cu
int launch_usckf(int pm, int mm, bool predict, bool update, const FilterArgs &a, cudaStream_t s);
bool usckf_shape_supported(int nk, int nl);
int launch_usckf_clone(int mode, const FilterArgs &a, cudaStream_t s);
int launch_usckf_set_measurement(int mode, const FilterArgs &a, cudaStream_t s);
// slb_msckf.cu
int launch_msckf_predict(int pm, const FilterArgs &a, cudaStream_t s);
int launch_msckf_update(int mm, const FilterArgs &a, cudaStream_t s);
int launch_msckf_update_ekf(int mm, const FilterArgs &a, cudaStream_t s);
// slb_check.cu
int launch_check_sigma_points(const slb_batch_s *h, int32_t *flags, double *diff, cudaStream_t s);
// slb_consistency.cu: out[6] += {NEES count, sum, sum of squares, NIS count, sum, sum of squares} (out zeroed by the caller)
int launch_consistency(const slb_batch_s *h, const double *truth, int t0, int n, double *nees, double *out, cudaStream_t s);
// slb_fusion.cu
int launch_fusion(int d, int64_t n, int op, const double *x1, const double *C1, const double *x2,
                  const double *C2, double *xo, double *Co, cudaStream_t s);

}  // namespace slb
