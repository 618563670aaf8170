/* slb.h -- C ABI of the B200-native batched sigma-point filter engine.
 *
 * This is the drop-in boundary for the hot path of jhidalgocarrio/slam-localization.  The
 * reference has no FFI: its boundary is the public member surface of header-only C++ class
 * templates.  Each entry point below names the reference member(s) it replaces (file:line,
 * relative to the reference root).  The host C++ facade in slam-localization_b200/facade/
 * re-creates those class surfaces (localization::Usckf / Msckf / DataModel, ukfom::ukf) on top
 * of exactly these symbols; INTEGRATION.md shows the binding a reference maintainer would add.
 *
 * Conventions
 *   - plain C types only; device pointers are `double*` obtained from cudaMalloc (or a torch
 *     tensor's data_ptr); `stream` is a cudaStream_t passed as void* (NULL = default stream).
 *   - every function returns 0 on success or a negative slb_error; nothing throws across the
 *     ABI.  Numerical trouble is never an error: it is recorded per instance in a status word
 *     (SLB_ST_* bits) that slb_status() summarises.
 *   - there is no CPU fallback.  Without a CUDA device slb_create fails with SLB_ERR_NO_DEVICE.
 *   - all arithmetic is IEEE double, like the reference's Eigen `double` path.
 *
 * State representation ("q-vector"): a manifold point is a flat array with 3 doubles per
 * vect<3> block and 4 doubles (w,x,y,z) per SO3 block, followed by plain feature scalars.
 * Tangent vectors / covariances use 3 DOF per block, in the same block order
 * (State.hpp:141-149,246-252,341-352,536-545; test/UKFoMUnitTest.cpp:31-35).
 */
#ifndef SLB_H_
#define SLB_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SLB_VERSION 100

typedef enum {
    SLB_OK = 0,
    SLB_ERR_INVALID = -1,    /* bad argument / unsupported combination            */
    SLB_ERR_NO_DEVICE = -2,  /* no CUDA device: the engine has no CPU fallback    */
    SLB_ERR_CUDA = -3,       /* a CUDA runtime call failed (see slb_last_error)   */
    SLB_ERR_ALLOC = -4,
    SLB_ERR_NCCL = -5
} slb_error;

/* Per-instance status bits (never abort the batch; reference behaviour in brackets). */
enum {
    SLB_ST_CHOL_FAIL = 1,   /* LLT pivot <= 0 [Eigen::LLT info() ignored, Usckf.hpp:537-538].
                               Usckf::update factors only the columns of Pk that can move h
                               (j < 36 + nk, rounded up to 4): a non-positive pivot beyond them is
                               neither computed nor flagged (the reference would write NaN into the
                               featuresk_l rows there); slb_check_sigma_points tests all of Pk      */
    SLB_ST_MEAN_NOCONV = 2, /* manifold mean hit max_it [assert(false), Usckf.hpp:620-624]     */
    SLB_ST_GATE_REJECT = 4, /* significance test rejected the update [Usckf.hpp:294]           */
    SLB_ST_NONFINITE = 8,   /* NaN/Inf met in the state                                        */
    SLB_ST_QR_ROWS = 16     /* Msckf EKF update: fewer measurement rows than DOF left after the
                               outlier removal [R.block(0,0,N,N) out of range, Msckf.hpp:808]  */
};
#define SLB_NSTATUS 5       /* number of status bits above */

/* Filter kinds (which reference class the batch stands for). */
enum {
    SLB_KIND_UKF = 1,   /* ukfom::ukf<state>            (test/UKFoMUnitTest.cpp:104-117)  */
    SLB_KIND_USCKF = 2, /* localization::Usckf<Aug,State> (Usckf.hpp:44-45)               */
    SLB_KIND_MSCKF = 3  /* localization::Msckf<Multi,State> (Msckf.hpp:40-41)             */
};

/* Fixed-DOF manifold layouts for SLB_KIND_UKF. */
enum {
    SLB_LAYOUT_POSE6 = 6,   /* vect3 pos, SO3 orient           (SensorState, State.hpp:242-252) */
    SLB_LAYOUT_MTK9 = 9     /* vect3 pos, SO3 orient, vect3 vel (test/UKFoMUnitTest.cpp:31-35)  */
};

/* Device model catalogue.  The reference takes arbitrary host functors f/h (Usckf.hpp:113-114,
 * 260-263); a GPU batch cannot call back into host code, so the models the reference ships in
 * its tests are compiled in and selected by id.  `u` is the per-instance control input. */
enum {
    /* process models */
    SLB_PM_UKFOM_IMU = 1,      /* test/UKFoMUnitTest.cpp:45-70 with orient = s.orient [+] w*dt;
                                  u = acc(3) gyro(3); layout MTK9                               */
    SLB_PM_UKFOM_IMU_REFBUG = 2, /* same, reproducing :53 (orient = identity [+] w*dt)            */
    SLB_PM_POSE6_ODOM = 3,     /* pos += R(q) v dt ; q = q*exp(w dt); u = v(3) w(3); POSE6      */
    SLB_PM_USCKF_TEST = 4,     /* test/UsckfUnitTest.cpp:34-49; u = velocity(3) angvel(3)       */
    SLB_PM_MSCKF_DELTAPOSE = 5,/* test/MsckfUnitTest.cpp:33-47; u = dp(3) dq(w,x,y,z) v(3) w(3) */
    /* measurement models */
    SLB_MM_GPS_POS = 101,      /* test/UKFoMUnitTest.cpp:82-85: z = pos (m = 3)                 */
    SLB_MM_USCKF_VO = 102,     /* test/UsckfUnitTest.cpp:62-86: featuresk moved by
                                  (statek [-] statek_i); m = nk                                 */
    SLB_MM_MSCKF_REPROJ = 103  /* builder-defined (the reference stops before update,
                                  test/MsckfUnitTest.cpp:215-232): pinhole reprojection of
                                  shared landmarks, feature f seen from clone f % k; m = 2*nfeat */
};

/* Cloning modes, Usckf.hpp:37-42 */
enum { SLB_STATEK = 1, SLB_STATEK_L = 2, SLB_STATEK_I = 3 };

/* Fields for slb_upload / slb_download (host side is always instance-major, dense). */
enum {
    SLB_FIELD_MU = 1,     /* batch x qdim q-vectors                              */
    SLB_FIELD_P = 2,      /* batch x N x N row-major covariances                 */
    SLB_FIELD_STATUS = 3, /* batch x int32 (download only; pass an int32_t*)     */
    SLB_FIELD_OUTLIERS = 4,/* batch x int32 outlier count of the last MSCKF update */
    SLB_FIELD_NIS = 5     /* batch x double NIS of the last UKF / USCKF update (download only, with
                             slb_set_nis_capture on; see there)                 */
};

typedef struct {
    int32_t kind;      /* SLB_KIND_*                                                     */
    int32_t layout;    /* SLB_LAYOUT_* for KIND_UKF; ignored otherwise                   */
    int32_t batch;     /* number of independent filter instances on this device          */
    int32_t nk, nl;    /* USCKF: featuresk.size(), featuresk_l.size() (State.hpp:539-540);
                          built shapes: nk in {3,6,9}, nl in {0,3,6,9}, nk + nl <= 12         */
    int32_t nclones;   /* MSCKF: sensorsk.size() (State.hpp:342)                         */
    int32_t device;    /* CUDA device ordinal                                            */
    int32_t reserved[9];
} slb_config;

typedef struct slb_batch_s *slb_handle;

/* ---- lifetime -------------------------------------------------------------------------- */
/* ctor of Usckf (Usckf.hpp:83) / Msckf (Msckf.hpp:80) / ukfom::ukf(mu,sigma): allocates the
 * device-resident batch; state is supplied with slb_upload. */
int slb_create(const slb_config *cfg, slb_handle *out);
int slb_destroy(slb_handle h);
const char *slb_last_error(void);
int slb_version(void);
int slb_dof(slb_handle h);   /* N: getDOF() (State.hpp:373-376,590-593) */
int slb_qdim(slb_handle h);  /* length of a q-vector                    */

/* ---- state access: muState()/PkAugmentedState() (Usckf.hpp:518-526), getPk()/setPk()
 *      (Msckf.hpp:386-395), ukf::mu()/sigma() ------------------------------------------------ */
/* count = k * (per-instance size): the first k instances are transferred (k = batch for all). */
int slb_upload(slb_handle h, int field, const void *host, size_t count, void *stream);
int slb_download(slb_handle h, int field, void *host, size_t count, void *stream);
/* Fleet initialisation: instance i <- instance (i % count) for i >= count, i.e. Monte-Carlo
 * replicas of the first `count` priors (new; the reference constructs one filter at a time). */
int slb_replicate(slb_handle h, int count, void *stream);
/* Raw device storage (engine-native layout, see DESIGN.md) for zero-copy consumers. */
int slb_device_ptr(slb_handle h, int field, void **dev);

/* ---- ukfom::ukf<state> ----------------------------------------------------------------- */
/* predict(g, R): sigma points -> g -> manifold mean -> cov + Q. u_dev: batch x nu (instance-
 * major), Q_dev: n x n row-major shared by the batch (batch x n x n with SLB_NOISE_Q_PER_INSTANCE, see
 * slb_set_noise_layout). */
int slb_ukf_predict(slb_handle h, int pm, const double *u_dev, double dt, const double *Q_dev,
                    void *stream);
/* update(z, h, R[, mt]): gate_dof = 0 accepts any Mahalanobis distance, 1..9 applies the 5%
 * chi-square table (Usckf.hpp:794-855). z_dev: batch x m, R_dev: m x m shared (batch x m x m
 * with SLB_NOISE_R_PER_INSTANCE, see slb_set_noise_layout). */
int slb_ukf_update(slb_handle h, int mm, const double *z_dev, const double *R_dev, int gate_dof,
                   void *stream);
/* predict immediately followed by update in one launch (one HBM round trip). */
int slb_ukf_step(slb_handle h, int pm, int mm, const double *u_dev, double dt,
                 const double *Q_dev, const double *z_dev, const double *R_dev, int gate_dof,
                 void *stream);
/* Same step with HOST buffers: copies u and z to the device, runs the step, copies the
 * posterior q-vectors back (mu_out_host: batch x qdim, may be NULL) and synchronises. */
int slb_ukf_step_host(slb_handle h, int pm, int mm, const double *u_host, double dt,
                      const double *Q_host, const double *z_host, const double *R_host,
                      int gate_dof, double *mu_out_host, void *stream);

/* Which part of the posterior q-vector the *_step_host entry points copy back: scalars [offset, offset +
 * count) of every instance, mu_out_host being batch x count.  Default: the whole q-vector (muState(),
 * Usckf.hpp:518).  (26, 13) on a USCKF batch is statek_i, what Usckf::muSingleState() returns by default
 * (Usckf.hpp:457-478); (0, 13) on an MSCKF batch is Msckf::muSingleState() (Msckf.hpp:356). */
int slb_set_output_slice(slb_handle h, int offset, int count);
/* Layout of the noise covariances that later device entry points receive on this handle.  0 (the default) = one
 * matrix shared by the batch, as before.  Q_PER_INSTANCE: Q_dev is batch x n x n row-major (instance i's matrix at
 * Q_dev + i*n*n; lower triangle read, like the shared Q).  R_PER_INSTANCE: R_dev is batch x m x m row-major.
 * Honoured by slb_ukf_predict/update/step (n = 6 or 9, m = 3), slb_usckf_predict/update/step (n = 12, m = nk),
 * slb_usckf_set_measurement (R: len x len per instance) and slb_msckf_predict (n = 12).  Like the reference, which
 * takes its noise per call and per object (Usckf::predict(f, Q), update(z, h, R), setMeasurement(mode, z, R)), a batch
 * of B then stands for B objects handed different covariances.  SLB_ERR_INVALID for flags outside 0..3 and for
 * R_PER_INSTANCE on an MSCKF handle (its update noise is shared).  While the flags are non-zero the *_step_host and
 * *_step_host_async entry points refuse to run: per-instance noise is device-resident only. */
enum { SLB_NOISE_Q_PER_INSTANCE = 1, SLB_NOISE_R_PER_INSTANCE = 2 };
int slb_set_noise_layout(slb_handle h, int flags);
/* NIS capture: the Mahalanobis distance m2 = nu^T S^-1 nu that update(z, h, R, mt) hands to the caller's `mt` functor
 * (Usckf.hpp:262,290-294).  on = 1 allocates batch doubles on the handle's device, filled with NaN; from then on every
 * update-bearing call (slb_ukf_update / step / step_host[_async], slb_usckf_update / step / step_host[_async]) rewrites
 * all of them with the m2 its gate was given, accepted or rejected, or NaN where the update stopped before forming it
 * (SLB_ST_CHOL_FAIL).  Predict-only calls leave them alone.  on = 0 stops writing and frees the array.  Read it with
 * slb_download(SLB_FIELD_NIS) or slb_device_ptr(SLB_FIELD_NIS), both SLB_ERR_INVALID while capture is off.
 * SLB_ERR_INVALID on an MSCKF handle: its update gates per feature and forms no whole-innovation distance. */
int slb_set_nis_capture(slb_handle h, int on);
/* Pipelined flavour: identical, but returns as soon as the step is enqueued on `stream` (no
 * synchronisation), so consecutive steps overlap their host<->device traffic with each other's
 * kernels.  The host buffers must stay valid (and mu_out_host unread) until slb_wait(h, stream);
 * pageable (not page-locked) buffers fall back to the synchronous behaviour.  Exists for all three
 * filter kinds (slb_usckf_step_host_async, slb_msckf_step_host_async below). */
int slb_ukf_step_host_async(slb_handle h, int pm, int mm, const double *u_host, double dt,
                            const double *Q_host, const double *z_host, const double *R_host,
                            int gate_dof, double *mu_out_host, void *stream);
/* Completes every step enqueued on `stream` by the *_step_host_async entry points. */
int slb_wait(slb_handle h, void *stream);

/* ---- localization::Usckf --------------------------------------------------------------- */
/* predict(f, Q) Usckf.hpp:107-244 */
int slb_usckf_predict(slb_handle h, int pm, const double *u_dev, double dt, const double *Q_dev,
                      void *stream);
/* update(z, h, R[, mt]) Usckf.hpp:246-308; z_dev: batch x m, R_dev: m x m shared (batch x m x m with
 * SLB_NOISE_R_PER_INSTANCE); predict's Q_dev: 12 x 12 (batch x 12 x 12 with SLB_NOISE_Q_PER_INSTANCE) */
int slb_usckf_update(slb_handle h, int mm, const double *z_dev, const double *R_dev,
                     int gate_dof, void *stream);
int slb_usckf_step(slb_handle h, int pm, int mm, const double *u_dev, double dt,
                   const double *Q_dev, const double *z_dev, const double *R_dev, int gate_dof,
                   void *stream);
int slb_usckf_step_host(slb_handle h, int pm, int mm, const double *u_host, double dt,
                        const double *Q_host, const double *z_host, const double *R_host,
                        int gate_dof, double *mu_out_host, void *stream);
int slb_usckf_step_host_async(slb_handle h, int pm, int mm, const double *u_host, double dt,
                              const double *Q_host, const double *z_host, const double *R_host,
                              int gate_dof, double *mu_out_host, void *stream);
/* cloning(mode) Usckf.hpp:391-433 */
int slb_usckf_clone(slb_handle h, int mode, void *stream);
/* setMeasurement(mode, z, R) Usckf.hpp:322-389; z_dev: batch x len, R_dev: len x len shared
 * (batch x len x len with SLB_NOISE_R_PER_INSTANCE).
 * len must equal the configured nk (mode STATEK) or nl (STATEK_L). */
int slb_usckf_set_measurement(slb_handle h, int mode, const double *z_dev, const double *R_dev,
                              void *stream);

/* ---- localization::Msckf --------------------------------------------------------------- */
/* predict(f, Q) Msckf.hpp:89-189; Q_dev: 12 x 12 shared (batch x 12 x 12 with SLB_NOISE_Q_PER_INSTANCE) */
int slb_msckf_predict(slb_handle h, int pm, const double *u_dev, double dt, const double *Q_dev,
                      void *stream);
/* update(z, h, R[, mt]) Msckf.hpp:196-277 (UKF flavour, per-feature 2-dof gate when gate != 0).
 * params_dev: model parameters shared by the batch (REPROJ: nfeat x 3 landmark coordinates);
 * z_dev: batch x m; R_dev: m x m shared.  The per-instance outlier count (the reference's
 * return value, :276) is kept in SLB_FIELD_OUTLIERS. */
int slb_msckf_update(slb_handle h, int mm, const double *params_dev, int m, const double *z_dev,
                     const double *R_dev, int gate, void *stream);

/* SURVEY 8(f) row f1 -- update(z, h, H, R[, mt]) Msckf.hpp:285-349, the EKF flavour: h also returns
 * its Jacobian H (m x N), removeOutliers works on the information matrix (:756-792, quirk Q6 and the
 * never-compacted `information` reproduced), reduceDimension compresses (H, innovation, R) through a
 * Householder QR (:794-816), then S = H P H^T + R, K = P H^T S^-1, Pk -= K S K^T, mu = mu [+] K nu.
 * Same arguments as slb_msckf_update; an instance left with fewer rows than DOF is flagged
 * SLB_ST_QR_ROWS and left unchanged. */
int slb_msckf_update_ekf(slb_handle h, int mm, const double *params_dev, int m, const double *z_dev,
                         const double *R_dev, int gate, void *stream);

/* predict + update with HOST buffers: u (batch x nu), z (batch x m) and the shared Q (12x12),
 * params (nparams doubles), R (m x m) are copied to the device, both kernels run, the posterior
 * q-vectors are copied back (mu_out_host: batch x qdim, may be NULL) and the stream is synchronised. */
int slb_msckf_step_host(slb_handle h, int pm, int mm, const double *u_host, double dt,
                        const double *Q_host, const double *params_host, int nparams, int m,
                        const double *z_host, const double *R_host, int gate, double *mu_out_host,
                        void *stream);

int slb_msckf_step_host_async(slb_handle h, int pm, int mm, const double *u_host, double dt,
                              const double *Q_host, const double *params_host, int nparams, int m,
                              const double *z_host, const double *R_host, int gate,
                              double *mu_out_host, void *stream);

/* ---- localization::DataModel<double,D> ---------------------------------------------------
 * fusion(data2) DataModel.hpp:48-60 over n independent pairs.  Instance-major device arrays:
 * x*: n x d, C*: n x d x d row-major.  d in {3, 6}.  Output may alias input 1 (in-place, like
 * the reference's data1.fusion(data2)). */
int slb_datamodel_fuse(int d, int64_t n, const double *x1, const double *C1, const double *x2,
                       const double *C2, double *xo, double *Co, void *stream);
/* operator+ / operator- DataModel.hpp:132-152 (both ADD the covariances). sign = +1 / -1 */
int slb_datamodel_addsub(int d, int64_t n, int sign, const double *x1, const double *C1,
                         const double *x2, const double *C2, double *xo, double *Co, void *stream);
/* Host-buffer variant of slb_datamodel_fuse (H2D, kernel, D2H, synchronise). */
int slb_datamodel_fuse_host(int d, int64_t n, const double *x1, const double *C1,
                            const double *x2, const double *C2, double *xo, double *Co);

/* ==== SURVEY section 8(f) "next" rows ======================================================= */

/* ---- f2: error-state EKF of src/filters/UsckfError.hpp (the Joseph-form variant of Usckf) ----
 * Instance-major device arrays holding what the reference object holds: mu = mu_state as 3 x 16
 * q-vector scalars (statek | statek_l | statek_i; per state pos vel quat(w,x,y,z) gbias abias, the
 * 15-DOF layout of :527-531), err = mu_error vectorised (n x 45), P = Pk_error dense row-major
 * (n x 45 x 45; the lower triangle is read, both are written). */
/* ekfPredict(F, Q) UsckfError.hpp:87-137.  F: n x 15 x 15 (per instance), Q: 15 x 15 shared. */
int slb_ekf_predict(int64_t n, double *err, double *P, const double *F, const double *Q, void *stream);
/* ekfUpdate(z, H, R[, mt]) UsckfError.hpp:322-384: Joseph-form covariance update + symmetrisation.
 * H: m x 45 shared, R: m x m shared, z: n x m.  gate 0 = accept any; otherwise the 5% chi-square
 * table with dof = m - 1 (the reference passes innovation.size()-1, :350).  ret (n x m) receives
 * the function's return value (zeros when accepted, the innovation when rejected), accepted (n)
 * the decision.  Like the reference only Pk_error changes.  m = 3. */
int slb_ekf_update(int64_t n, int m, const double *mu, double *P, const double *z, const double *H,
                   const double *R, int gate, double *ret, int32_t *accepted, void *stream);
/* ekfSingleUpdate(z, H, R[, mt]) UsckfError.hpp:489-571 on the statek_i block; H: m x 15.  The
 * corrections are applied to mu_state.statek_i whatever the gate says (:553-568). m = 3. */
int slb_ekf_single_update(int64_t n, int m, double *mu, const double *err, double *P, const double *z,
                          const double *H, const double *R, int gate, int32_t *accepted, void *stream);
/* cloning() UsckfError.hpp:573-603 */
int slb_ekf_clone(int64_t n, double *mu, double *err, double *P, void *stream);

/* ---- f3: DataModel<double,3>::safeFusion(data2) DataModel.hpp:62-130 (d = 3 only, :104) ------ */
int slb_datamodel_safe_fuse(int64_t n, const double *x1, const double *C1, const double *x2,
                            const double *C2, double *xo, double *Co, void *stream);

/* ---- f4: the producers of the filters' odometry input ----------------------------------------
 * Poses are pos(3) quat(w,x,y,z); covariances are 6 x 6 over [r t], rotation first
 * (Transform.hpp:48-60).  result = t2 * t1, TransformWithUncertainty::operator* Transform.cpp:215-254
 * (both operands uncertain). */
int slb_transform_compose(int64_t n, const double *pose2, const double *cov2, const double *pose1,
                          const double *cov1, double *pose_out, double *cov_out, void *stream);
/* DeadReckon::updatePose(delta_t, cartesianVelocities, cartesianVelCov, prevPose, postPose)
 * DeadReckon.hpp:30-79 (with updateAttitude :246-286).  vel0 / vel1: n x 6 (linear, angular) at the
 * current and the previous sample; velcov: 6 x 6 shared.  post = prev * delta; the returned
 * deltaPose goes to delta_pose / delta_cov. */
int slb_deadreckon_update_pose(int64_t n, double dt, const double *vel0, const double *vel1,
                               const double *velcov, const double *prev_pose, const double *prev_cov,
                               double *post_pose, double *post_cov, double *delta_pose,
                               double *delta_cov, void *stream);

/* ---- device buffers for callers without a CUDA binding (cgo / JNI / ctypes, the C++ facade) ---- */
int slb_dev_alloc(size_t bytes, void **dev);
int slb_dev_free(void *dev);
/* kind: 1 host->device, 2 device->host, 3 device->device; synchronises the stream for kind 2. */
int slb_dev_copy(void *dst, const void *src, size_t bytes, int kind, void *stream);

/* ---- diagnostics ----------------------------------------------------------------------- */
/* counts[0..3] = instances with CHOL_FAIL / MEAN_NOCONV / GATE_REJECT / NONFINITE set. */
int slb_status(slb_handle h, int64_t counts[4], void *stream);
/* The same for the first nbits <= SLB_NSTATUS status bits (counts[4] = QR_ROWS). */
int slb_status_ex(slb_handle h, int64_t *counts, int nbits, void *stream);
int slb_clear_status(slb_handle h, void *stream);
/* Ensemble statistics of the instance means over this device's shard (new; no reference
 * counterpart): out = { count, sum x[nv], sum x x^T[nv*nv] } with x = the vect<3> blocks and
 * the SO3 log of every block of the q-vector; out_dev has 1 + nv + nv*nv doubles, nv = N.
 * Multi-GPU callers all-reduce out_dev (NCCL sum) -- see bench.py. */
int slb_ensemble_stats(slb_handle h, double *out_dev, void *stream);
/* The same, merged over the ranks of an NCCL communicator (SURVEY 8e: the only collective of the path, end of
 * run): slb_ensemble_stats on this device's shard, then ncclAllReduce(sum, double) of the 1 + nv + nv*nv
 * values in place on `stream`.  nccl_comm is an ncclComm_t passed as void* (NULL = this shard only).  NCCL is
 * resolved at run time (dlopen libnccl.so.2); SLB_ERR_NCCL if it is missing or a call fails. */
int slb_gather_stats(slb_handle h, void *nccl_comm, double *out_dev, void *stream);
/* Filter consistency (new; the reference has no counterpart -- its user would download every Pk and invert it):
 * out_dev: 6 doubles, overwritten with {NEES count, sum, sum of squares, NIS count, sum, sum of squares} over this shard.
 * truth_dev: batch x qdim q-vectors, instance-major dense (slb_upload's SLB_FIELD_MU format), or NULL = no NEES, in
 * which case t0 = n = 0 and nees_dev is not written.  [t0, t0 + n): the tangent coordinates covered, in
 * slb_ensemble_stats' vectorisation (3 per 3-DOF block, then the feature scalars); neither end may cut a 3-DOF block.
 * Per instance NEES = e^T P_sub^-1 e with e = truth [-] mu (MTK: log(mu_q^-1 truth_q) on SO3 blocks, a difference
 * elsewhere) and P_sub = P[t0:t0+n, t0:t0+n] the marginal covariance, from a Cholesky factorisation of P_sub; a
 * non-positive or non-finite pivot or a non-finite e gives NaN and leaves the instance out of the count (status bits
 * are not touched).  nees_dev: batch doubles or NULL.  The NIS triplet sums the finite entries of the captured NIS
 * (slb_set_nis_capture), zeros when capture is off.  SLB_ERR_INVALID for a bad range, before any device work. */
int slb_consistency_stats(slb_handle h, const double *truth_dev, int t0, int n, double *nees_dev, double *out_dev,
                          void *stream);
/* The same, merged over the ranks of an NCCL communicator: slb_consistency_stats on this shard, then
 * ncclAllReduce(sum, double) of the 6 values in place on `stream` (nccl_comm NULL = this shard only). */
int slb_gather_consistency(slb_handle h, void *nccl_comm, const double *truth_dev, int t0, int n, double *nees_dev,
                           double *out_dev, void *stream);
/* Communicator helpers for callers without an NCCL binding of their own (ctypes, cgo, the C++ facade):
 * rank 0 calls slb_nccl_unique_id (id128: 128 bytes) and ships the bytes to the other ranks by any means,
 * every rank then calls slb_nccl_comm_init with its rank and CUDA device. */
int slb_nccl_unique_id(void *id128);
int slb_nccl_comm_init(void **comm, int nranks, const void *id128, int rank, int device);
int slb_nccl_comm_destroy(void *comm);

/* checkSigmaPoints() Usckf.hpp:769-789 / Msckf.hpp:818-838 for every instance of a USCKF / MSCKF batch:
 * sigma points of (mu_state, Pk), their manifold mean muX and covariance Pktest.  The reference asserts
 * max|Pktest - Pk| <= 1e-6 and mu_state == muX; the batch reports per instance
 *   flags_dev[i] (int32): bit 0 covariance off by more than 1e-6, bit 1 mean moved by more than 1e-12 (tangent
 *                         space, inf-norm; the reference's exact == is rounding noise), bit 2 LLT of Pk failed
 *   diff_dev[2i], [2i+1]: max|Pktest - Pk| and |muX [-] mu|_inf (diff_dev may be NULL). */
int slb_check_sigma_points(slb_handle h, int32_t *flags_dev, double *diff_dev, void *stream);

/* Measures the device's FP64 FMA rate (TFLOP/s, FMA = 2) with a register-resident DFMA kernel:
 * the roofline denominator for the FP64-bound configs (MEASURED_PEAKS.json has no FP64 entry). */
int slb_bench_fp64_peak(double *tflops_out);
/* Number of kernels this library has launched since load (bench.py's gpu_launches). */
int64_t slb_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* SLB_H_ */
