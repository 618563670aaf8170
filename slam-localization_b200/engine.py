"""ctypes binding of csrc/libslb.so -- the C ABI of include/slb.h -- plus thin host-side classes that
mirror the reference's filter surface (Usckf / Msckf / ukfom::ukf / DataModel) for batches.

torch is used for device memory and streams only.  There is NO CPU fallback: importing works
anywhere (so the symbol table can be checked), but every compute call needs the CUDA library and
a CUDA device and fails loudly otherwise."""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("SLB_LIB") or os.path.join(_HERE, "csrc", "libslb.so")   # SLB_LIB: experiment builds of the library

# ---- ids of include/slb.h ------------------------------------------------------------------------
KIND_UKF, KIND_USCKF, KIND_MSCKF = 1, 2, 3
LAYOUT_POSE6, LAYOUT_MTK9 = 6, 9
PM_UKFOM_IMU, PM_UKFOM_IMU_REFBUG, PM_POSE6_ODOM, PM_USCKF_TEST, PM_MSCKF_DELTAPOSE = 1, 2, 3, 4, 5
MM_GPS_POS, MM_USCKF_VO, MM_MSCKF_REPROJ = 101, 102, 103
STATEK, STATEK_L, STATEK_I = 1, 2, 3
FIELD_MU, FIELD_P, FIELD_STATUS, FIELD_OUTLIERS, FIELD_NIS = 1, 2, 3, 4, 5
ST_CHOL_FAIL, ST_MEAN_NOCONV, ST_GATE_REJECT, ST_NONFINITE, ST_QR_ROWS = 1, 2, 4, 8, 16
NSTATUS = 5
NOISE_Q_PER_INSTANCE, NOISE_R_PER_INSTANCE = 1, 2

EXPORTS = [
    "slb_version", "slb_last_error", "slb_create", "slb_destroy", "slb_dof", "slb_qdim", "slb_upload",
    "slb_download", "slb_device_ptr", "slb_ukf_predict", "slb_ukf_update", "slb_ukf_step", "slb_ukf_step_host",
    "slb_usckf_predict", "slb_usckf_update", "slb_usckf_step", "slb_usckf_step_host", "slb_usckf_clone",
    "slb_usckf_set_measurement", "slb_msckf_predict", "slb_msckf_update", "slb_datamodel_fuse",
    "slb_datamodel_addsub", "slb_datamodel_fuse_host", "slb_status", "slb_status_ex", "slb_clear_status", "slb_ensemble_stats",
    "slb_launch_count", "slb_bench_fp64_peak", "slb_replicate", "slb_dev_alloc", "slb_dev_free", "slb_dev_copy",
    "slb_msckf_step_host", "slb_ekf_predict", "slb_ekf_update", "slb_ekf_single_update", "slb_ekf_clone",
    "slb_datamodel_safe_fuse", "slb_msckf_update_ekf", "slb_transform_compose", "slb_deadreckon_update_pose",
    "slb_ukf_step_host_async", "slb_usckf_step_host_async", "slb_msckf_step_host_async", "slb_wait",
    "slb_set_output_slice", "slb_set_noise_layout", "slb_check_sigma_points", "slb_gather_stats", "slb_nccl_unique_id", "slb_nccl_comm_init", "slb_nccl_comm_destroy",
    "slb_set_nis_capture", "slb_consistency_stats", "slb_gather_consistency",
]


class SlbConfig(C.Structure):
    _fields_ = [("kind", C.c_int32), ("layout", C.c_int32), ("batch", C.c_int32), ("nk", C.c_int32),
                ("nl", C.c_int32), ("nclones", C.c_int32), ("device", C.c_int32), ("reserved", C.c_int32 * 9)]


class SlbError(RuntimeError):
    pass


_lib = None


def lib():
    """Load libslb.so; raises if it has not been built (no silent fallback)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise SlbError("CUDA library %s is missing: run __graft_entry__.build() (there is no CPU fallback)" % LIB_PATH)
        L = C.CDLL(LIB_PATH)
        vp, dp, i32, i64, dbl = C.c_void_p, C.c_void_p, C.c_int, C.c_int64, C.c_double
        L.slb_last_error.restype = C.c_char_p
        L.slb_launch_count.restype = C.c_int64
        L.slb_create.argtypes = [C.POINTER(SlbConfig), C.POINTER(vp)]
        L.slb_destroy.argtypes = [vp]
        L.slb_dof.argtypes = [vp]
        L.slb_qdim.argtypes = [vp]
        L.slb_upload.argtypes = [vp, i32, vp, C.c_size_t, vp]
        L.slb_download.argtypes = [vp, i32, vp, C.c_size_t, vp]
        L.slb_device_ptr.argtypes = [vp, i32, C.POINTER(vp)]
        L.slb_replicate.argtypes = [vp, i32, vp]
        L.slb_ukf_predict.argtypes = [vp, i32, dp, dbl, dp, vp]
        L.slb_ukf_update.argtypes = [vp, i32, dp, dp, i32, vp]
        L.slb_ukf_step.argtypes = [vp, i32, i32, dp, dbl, dp, dp, dp, i32, vp]
        L.slb_ukf_step_host.argtypes = [vp, i32, i32, dp, dbl, dp, dp, dp, i32, dp, vp]
        L.slb_usckf_predict.argtypes = [vp, i32, dp, dbl, dp, vp]
        L.slb_usckf_update.argtypes = [vp, i32, dp, dp, i32, vp]
        L.slb_usckf_step.argtypes = [vp, i32, i32, dp, dbl, dp, dp, dp, i32, vp]
        L.slb_usckf_step_host.argtypes = [vp, i32, i32, dp, dbl, dp, dp, dp, i32, dp, vp]
        L.slb_ukf_step_host_async.argtypes = L.slb_ukf_step_host.argtypes
        L.slb_usckf_step_host_async.argtypes = L.slb_usckf_step_host.argtypes
        L.slb_wait.argtypes = [vp, vp]
        L.slb_set_output_slice.argtypes = [vp, i32, i32]
        L.slb_set_noise_layout.argtypes = [vp, i32]
        L.slb_set_nis_capture.argtypes = [vp, i32]
        L.slb_consistency_stats.argtypes = [vp, dp, i32, i32, dp, dp, vp]
        L.slb_gather_consistency.argtypes = [vp, vp, dp, i32, i32, dp, dp, vp]
        L.slb_check_sigma_points.argtypes = [vp, vp, vp, vp]
        L.slb_gather_stats.argtypes = [vp, vp, dp, vp]
        L.slb_nccl_unique_id.argtypes = [vp]
        L.slb_nccl_comm_init.argtypes = [C.POINTER(vp), i32, vp, i32, i32]
        L.slb_nccl_comm_destroy.argtypes = [vp]
        L.slb_usckf_clone.argtypes = [vp, i32, vp]
        L.slb_usckf_set_measurement.argtypes = [vp, i32, dp, dp, vp]
        L.slb_msckf_predict.argtypes = [vp, i32, dp, dbl, dp, vp]
        L.slb_msckf_update.argtypes = [vp, i32, dp, i32, dp, dp, i32, vp]
        L.slb_msckf_update_ekf.argtypes = [vp, i32, dp, i32, dp, dp, i32, vp]
        L.slb_msckf_step_host.argtypes = [vp, i32, i32, dp, dbl, dp, dp, i32, i32, dp, dp, i32, dp, vp]
        L.slb_msckf_step_host_async.argtypes = L.slb_msckf_step_host.argtypes
        L.slb_datamodel_fuse.argtypes = [i32, i64, dp, dp, dp, dp, dp, dp, vp]
        L.slb_datamodel_addsub.argtypes = [i32, i64, i32, dp, dp, dp, dp, dp, dp, vp]
        L.slb_datamodel_fuse_host.argtypes = [i32, i64, dp, dp, dp, dp, dp, dp]
        L.slb_ekf_predict.argtypes = [i64, dp, dp, dp, dp, vp]
        L.slb_ekf_update.argtypes = [i64, i32, dp, dp, dp, dp, dp, i32, dp, vp, vp]
        L.slb_ekf_single_update.argtypes = [i64, i32, dp, dp, dp, dp, dp, dp, i32, vp, vp]
        L.slb_ekf_clone.argtypes = [i64, dp, dp, dp, vp]
        L.slb_datamodel_safe_fuse.argtypes = [i64, dp, dp, dp, dp, dp, dp, vp]
        L.slb_transform_compose.argtypes = [i64, dp, dp, dp, dp, dp, dp, vp]
        L.slb_deadreckon_update_pose.argtypes = [i64, dbl, dp, dp, dp, dp, dp, dp, dp, dp, dp, vp]
        L.slb_status.argtypes = [vp, C.POINTER(C.c_int64), vp]
        L.slb_status_ex.argtypes = [vp, C.POINTER(C.c_int64), i32, vp]
        L.slb_clear_status.argtypes = [vp, vp]
        L.slb_ensemble_stats.argtypes = [vp, dp, vp]
        _lib = L
    return _lib


def check(rc):
    if rc != 0:
        raise SlbError("slb error %d: %s" % (rc, lib().slb_last_error().decode()))


def fp64_peak_tflops():
    _torch()
    v = C.c_double(0.0)
    check(lib().slb_bench_fp64_peak(C.byref(v)))
    return v.value


def launch_count():
    return int(lib().slb_launch_count())


def _torch():
    import torch
    if not torch.cuda.is_available():
        raise SlbError("no CUDA device: the engine has no CPU fallback")
    return torch


def _stream():
    return C.c_void_p(_torch().cuda.current_stream().cuda_stream)


def _hp(a):
    return a.ctypes.data_as(C.c_void_p)


def _h(a, dtype=np.float64):
    return np.ascontiguousarray(a, dtype=dtype)


class DeviceArray:
    """A float64 torch tensor on the current device, passed to the C ABI as a raw pointer."""

    def __init__(self, host=None, shape=None):
        torch = _torch()
        if host is not None:
            self.t = torch.from_numpy(_h(host)).cuda()
        else:
            self.t = torch.empty(shape, dtype=torch.float64, device="cuda")

    @property
    def ptr(self):
        return C.c_void_p(self.t.data_ptr())

    def numpy(self):
        return self.t.cpu().numpy()


def dev(a):
    """numpy -> a fresh device copy; DeviceArray -> itself; torch tensor (CUDA, or page-locked host memory, which the
    kernels can read in place through unified addressing) -> wrapped without a copy."""
    if isinstance(a, DeviceArray):
        return a
    if not isinstance(a, np.ndarray):
        torch = _torch()
        if isinstance(a, torch.Tensor):
            if not (a.is_cuda or a.is_pinned()):
                raise SlbError("host tensors must be page-locked (pin_memory) to be passed without a copy")
            w = DeviceArray.__new__(DeviceArray)
            w.t = a.contiguous()
            return w
    return DeviceArray(a)


class Batch:
    """A device-resident batch of filter instances (slb_handle)."""

    def __init__(self, kind, batch, layout=0, nk=0, nl=0, nclones=0, device=None):
        torch = _torch()
        cfg = SlbConfig()
        cfg.kind, cfg.layout, cfg.batch, cfg.nk, cfg.nl, cfg.nclones = kind, layout, batch, nk, nl, nclones
        cfg.device = torch.cuda.current_device() if device is None else device
        self.h = C.c_void_p()
        check(lib().slb_create(C.byref(cfg), C.byref(self.h)))
        self.B = batch
        self.N = lib().slb_dof(self.h)
        self.QD = lib().slb_qdim(self.h)
        self.kind, self.nk, self.nl, self.k = kind, nk, nl, nclones
        self.noise = 0   # slb_set_noise_layout flags of the handle

    def close(self):
        if self.h:
            lib().slb_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # state access: muState() / Pk (Usckf.hpp:518-526, Msckf.hpp:376-395)
    def set_state(self, mu, P, replicate=False):
        """Upload means / covariances.  With replicate=True only the first len(mu) instances are given and
        the rest of the batch is filled with copies (instance i <- i % len(mu))."""
        mu, P = _h(mu), _h(P)
        k = mu.shape[0]
        assert (k == self.B or replicate) and k <= self.B
        assert mu.shape == (k, self.QD) and P.shape == (k, self.N, self.N), (mu.shape, P.shape)
        check(lib().slb_upload(self.h, FIELD_MU, _hp(mu), mu.size, _stream()))
        check(lib().slb_upload(self.h, FIELD_P, _hp(P), P.size, _stream()))
        if k < self.B:
            check(lib().slb_replicate(self.h, k, _stream()))

    def mu(self, first=None):
        k = self.B if first is None else first
        out = np.empty((k, self.QD))
        check(lib().slb_download(self.h, FIELD_MU, _hp(out), out.size, _stream()))
        return out

    def P(self, first=None):
        k = self.B if first is None else first
        out = np.empty((k, self.N, self.N))
        check(lib().slb_download(self.h, FIELD_P, _hp(out), out.size, _stream()))
        return out

    def status(self):
        out = np.empty(self.B, np.int32)
        check(lib().slb_download(self.h, FIELD_STATUS, _hp(out), out.size, _stream()))
        return out

    def outliers(self):
        out = np.empty(self.B, np.int32)
        check(lib().slb_download(self.h, FIELD_OUTLIERS, _hp(out), out.size, _stream()))
        return out

    def status_counts(self):
        """Instances with CHOL_FAIL / MEAN_NOCONV / GATE_REJECT / NONFINITE / QR_ROWS set (all SLB_NSTATUS bits)."""
        c = (C.c_int64 * NSTATUS)()
        check(lib().slb_status_ex(self.h, c, NSTATUS, _stream()))
        return list(c)

    def set_output_slice(self, offset, count):
        """Part of the posterior q-vector step_host copies back (default: all); e.g. (26, 13) = statek_i of a USCKF."""
        check(lib().slb_set_output_slice(self.h, offset, count))

    def set_noise_layout(self, flags):
        """slb_set_noise_layout: NOISE_Q_PER_INSTANCE / NOISE_R_PER_INSTANCE make the device entry points read Q / R as
        batch x n x n arrays (one matrix per instance); 0 = one matrix shared by the batch.  The filter methods call it
        themselves from the shapes of the Q / R they are given."""
        check(lib().slb_set_noise_layout(self.h, flags))
        self.noise = flags

    def _noise_bit(self, name, a, n, bit):
        """The layout bit a noise matrix asks for: (n, n) is shared by the batch, (B, n, n) one matrix per instance."""
        shape = tuple(a.t.shape) if isinstance(a, DeviceArray) else tuple(a.shape) if hasattr(a, "shape") else np.shape(a)
        if shape == (n, n):
            return 0
        if shape == (self.B, n, n):
            return bit
        raise ValueError("%s must have shape (%d, %d) (shared by the batch) or (%d, %d, %d) (one per instance), got %s"
                         % (name, n, n, self.B, n, n, shape))

    def _use_noise(self, Q=None, n=0, R=None, m=0):
        """Checks the shapes of Q (n x n) / R (m x m) and sets the handle's noise layout to what they ask for (the bit of
        a matrix that is not passed is left as it is)."""
        flags = self.noise
        if Q is not None:
            flags = (flags & ~NOISE_Q_PER_INSTANCE) | self._noise_bit("Q", Q, n, NOISE_Q_PER_INSTANCE)
        if R is not None:
            flags = (flags & ~NOISE_R_PER_INSTANCE) | self._noise_bit("R", R, m, NOISE_R_PER_INSTANCE)
        if flags != self.noise:
            self.set_noise_layout(flags)

    def _host_noise(self, Q, n, R, m):
        """The host-buffer steps take shared noise only (per-instance noise is device-resident, slb_set_noise_layout): an
        array holding batch x n x n values is refused, anything else is passed through as before (n x n read)."""
        if self.B > 1 and (np.size(Q) == self.B * n * n or np.size(R) == self.B * m * m):
            raise ValueError("step_host takes Q and R shared by the batch; per-instance noise needs the device entry points")
        if self.noise:
            self.set_noise_layout(0)

    def wait(self):
        """Completes the steps enqueued with step_host(..., wait=False) on the current stream."""
        check(lib().slb_wait(self.h, _stream()))

    def clear_status(self):
        check(lib().slb_clear_status(self.h, _stream()))

    def ensemble_stats(self, out=None):
        out = out if out is not None else DeviceArray(shape=(1 + self.N + self.N * self.N,))
        check(lib().slb_ensemble_stats(self.h, out.ptr, _stream()))
        return out

    def gather_stats(self, comm=None, out=None):
        """slb_gather_stats: this shard's (count, sum x, sum x x^T) all-reduced over an NcclComm (None: local only)."""
        out = out if out is not None else DeviceArray(shape=(1 + self.N + self.N * self.N,))
        check(lib().slb_gather_stats(self.h, comm.c if comm is not None else None, out.ptr, _stream()))
        return out

    def set_nis_capture(self, on):
        """slb_set_nis_capture: while on, every update-bearing call stores each instance's Mahalanobis distance
        m2 = nu^T S^-1 nu (what the reference hands to `mt`), NaN where the update failed before forming it."""
        check(lib().slb_set_nis_capture(self.h, 1 if on else 0))

    def nis(self):
        """The captured NIS of the last update, (B,) float64 (SlbError while capture is off)."""
        out = np.empty(self.B)
        check(lib().slb_download(self.h, FIELD_NIS, _hp(out), out.size, _stream()))
        return out

    def _consistency(self, fn, comm, truth, t0, n, nees):
        if truth is None:
            t, n = None, 0 if n is None else n
        else:
            t = dev(truth)
            if tuple(t.t.shape) != (self.B, self.QD):
                raise ValueError("truth must have shape (%d, %d), got %s" % (self.B, self.QD, tuple(t.t.shape)))
            n = self.N - t0 if n is None else n
        out = DeviceArray(shape=(6,))
        ne = DeviceArray(shape=(self.B,)) if nees else None
        args = (t.ptr if t is not None else None, t0, n, ne.ptr if ne is not None else None, out.ptr, _stream())
        check(fn(self.h, *args) if comm is False else fn(self.h, comm.c if comm is not None else None, *args))
        return (out.numpy(), ne.numpy()) if nees else out.numpy()

    def consistency_stats(self, truth=None, t0=0, n=None, nees=False):
        """slb_consistency_stats: {NEES count, sum, sum of squares, NIS count, sum, sum of squares} over this batch.
        truth: (B, qdim) q-vectors (None = NIS only); [t0, t0 + n) the tangent coordinates of the NEES (n=None: to the
        end of the state).  nees=True also returns the per-instance NEES, NaN where P_sub is not positive definite."""
        return self._consistency(lib().slb_consistency_stats, False, truth, t0, n, nees)

    def gather_consistency(self, comm=None, truth=None, t0=0, n=None, nees=False):
        """slb_gather_consistency: consistency_stats all-reduced over an NcclComm (None: this shard only)."""
        return self._consistency(lib().slb_gather_consistency, comm, truth, t0, n, nees)

    def check_sigma_points(self):
        """checkSigmaPoints() (Usckf.hpp:769-789, Msckf.hpp:818-838): returns (flags[B] int32, diff[B, 2])."""
        torch = _torch()
        flags = torch.zeros(self.B, dtype=torch.int32, device="cuda")
        diff = DeviceArray(shape=(self.B, 2))
        check(lib().slb_check_sigma_points(self.h, C.c_void_p(flags.data_ptr()), diff.ptr, _stream()))
        return flags.cpu().numpy(), diff.numpy()


class NcclComm:
    """An ncclComm_t created through the C ABI (slb_nccl_unique_id / slb_nccl_comm_init).  `exchange(bytes_or_None)`
    ships rank 0's 128-byte unique id to every rank (e.g. a torch.distributed broadcast)."""

    def __init__(self, rank, world, exchange, device=None):
        torch = _torch()
        ident = (C.c_ubyte * 128)()
        if rank == 0:
            check(lib().slb_nccl_unique_id(ident))
        raw = exchange(bytes(ident) if rank == 0 else None)
        ident = (C.c_ubyte * 128).from_buffer_copy(raw)
        self.c = C.c_void_p()
        dev = torch.cuda.current_device() if device is None else device
        check(lib().slb_nccl_comm_init(C.byref(self.c), world, ident, rank, dev))

    def close(self):
        if self.c:
            lib().slb_nccl_comm_destroy(self.c)
            self.c = C.c_void_p()


class Ukf(Batch):
    """Batch of ukfom::ukf<state> (test/UKFoMUnitTest.cpp:104-117): predict(g,Q), update(z,h,R)."""

    def __init__(self, batch, layout=LAYOUT_MTK9, device=None):
        super().__init__(KIND_UKF, batch, layout=layout, device=device)

    def predict(self, pm, u, dt, Q):
        """Q: (n, n) shared by the batch or (batch, n, n) one per instance."""
        self._use_noise(Q=Q, n=self.N)
        u, Q = dev(u), dev(Q)
        check(lib().slb_ukf_predict(self.h, pm, u.ptr, dt, Q.ptr, _stream()))

    def update(self, mm, z, R, gate_dof=0):
        """R: (3, 3) shared by the batch or (batch, 3, 3) one per instance."""
        self._use_noise(R=R, m=3)
        z, R = dev(z), dev(R)
        check(lib().slb_ukf_update(self.h, mm, z.ptr, R.ptr, gate_dof, _stream()))

    def step(self, pm, mm, u, dt, Q, z, R, gate_dof=0):
        self._use_noise(Q=Q, n=self.N, R=R, m=3)
        u, Q, z, R = dev(u), dev(Q), dev(z), dev(R)
        check(lib().slb_ukf_step(self.h, pm, mm, u.ptr, dt, Q.ptr, z.ptr, R.ptr, gate_dof, _stream()))

    def step_host(self, pm, mm, u, dt, Q, z, R, gate_dof=0, mu_out=None, wait=True):
        """u, z, Q, R are HOST arrays (numpy or pinned torch); returns/fills the posterior means.  wait=False is the
        pipelined flavour (slb_ukf_step_host_async): call .wait() before touching the buffers again."""
        self._host_noise(Q, self.N, R, 3)
        fn = lib().slb_ukf_step_host if wait else lib().slb_ukf_step_host_async
        check(fn(self.h, pm, mm, _ptr_of(u), dt, _ptr_of(Q), _ptr_of(z), _ptr_of(R), gate_dof,
                 _ptr_of(mu_out) if mu_out is not None else None, _stream()))


class Usckf(Batch):
    """Batch of localization::Usckf<AugmentedState,State> (Usckf.hpp)."""

    def __init__(self, batch, nk=3, nl=9, device=None):
        super().__init__(KIND_USCKF, batch, nk=nk, nl=nl, device=device)

    def predict(self, pm, u, dt, Q):
        """Q: (12, 12) shared by the batch or (batch, 12, 12) one per instance."""
        self._use_noise(Q=Q, n=12)
        u, Q = dev(u), dev(Q)
        check(lib().slb_usckf_predict(self.h, pm, u.ptr, dt, Q.ptr, _stream()))

    def update(self, mm, z, R, gate_dof=0):
        """R: (nk, nk) shared by the batch or (batch, nk, nk) one per instance."""
        self._use_noise(R=R, m=self.nk)
        z, R = dev(z), dev(R)
        check(lib().slb_usckf_update(self.h, mm, z.ptr, R.ptr, gate_dof, _stream()))

    def step(self, pm, mm, u, dt, Q, z, R, gate_dof=0):
        self._use_noise(Q=Q, n=12, R=R, m=self.nk)
        u, Q, z, R = dev(u), dev(Q), dev(z), dev(R)
        check(lib().slb_usckf_step(self.h, pm, mm, u.ptr, dt, Q.ptr, z.ptr, R.ptr, gate_dof, _stream()))

    def step_host(self, pm, mm, u, dt, Q, z, R, gate_dof=0, mu_out=None, wait=True):
        self._host_noise(Q, 12, R, self.nk)
        fn = lib().slb_usckf_step_host if wait else lib().slb_usckf_step_host_async
        check(fn(self.h, pm, mm, _ptr_of(u), dt, _ptr_of(Q), _ptr_of(z), _ptr_of(R), gate_dof,
                 _ptr_of(mu_out) if mu_out is not None else None, _stream()))

    def cloning(self, mode):
        check(lib().slb_usckf_clone(self.h, mode, _stream()))

    def set_measurement(self, mode, z, R):
        """R: (len, len) shared by the batch or (batch, len, len) one per instance, len = nk (STATEK) or nl (STATEK_L)."""
        self._use_noise(R=R, m=self.nk if mode == STATEK else self.nl)
        z, R = dev(z), dev(R)
        check(lib().slb_usckf_set_measurement(self.h, mode, z.ptr, R.ptr, _stream()))


class Msckf(Batch):
    """Batch of localization::Msckf<MultiState,State> (Msckf.hpp), UKF-flavoured update."""

    def __init__(self, batch, nclones=10, device=None):
        super().__init__(KIND_MSCKF, batch, nclones=nclones, device=device)

    def predict(self, pm, u, dt, Q):
        """Q: (12, 12) shared by the batch or (batch, 12, 12) one per instance."""
        self._use_noise(Q=Q, n=12)
        u, Q = dev(u), dev(Q)
        check(lib().slb_msckf_predict(self.h, pm, u.ptr, dt, Q.ptr, _stream()))

    def update(self, mm, params, z, R, gate=True):
        params, z, R = dev(params), dev(z), dev(R)
        m = z.t.shape[1]
        check(lib().slb_msckf_update(self.h, mm, params.ptr, m, z.ptr, R.ptr, int(gate), _stream()))

    def update_ekf(self, mm, params, z, R, gate=True):
        """update(z, h, H, R[, mt]) -- the EKF flavour with QR compression (Msckf.hpp:285-349)."""
        params, z, R = dev(params), dev(z), dev(R)
        m = z.t.shape[1]
        check(lib().slb_msckf_update_ekf(self.h, mm, params.ptr, m, z.ptr, R.ptr, int(gate), _stream()))

    def step_host(self, pm, mm, u, dt, Q, params, z, R, gate=True, mu_out=None, wait=True):
        """predict + update with HOST arrays (numpy or pinned torch); fills the posterior means."""
        m = z.shape[1]
        self._host_noise(Q, 12, R, m)
        nparams = int(np.prod(params.shape))
        fn = lib().slb_msckf_step_host if wait else lib().slb_msckf_step_host_async
        check(fn(self.h, pm, mm, _ptr_of(u), dt, _ptr_of(Q), _ptr_of(params), nparams, m, _ptr_of(z), _ptr_of(R), int(gate),
                 _ptr_of(mu_out) if mu_out is not None else None, _stream()))


def _ptr_of(a):
    if a is None:
        return None
    if isinstance(a, np.ndarray):
        assert a.dtype == np.float64 and a.flags["C_CONTIGUOUS"]
        return _hp(a)
    return C.c_void_p(a.data_ptr())  # torch tensor (pinned host or device)


class DataModel:
    """localization::DataModel<double,D> over n independent estimates (DataModel.hpp)."""

    @staticmethod
    def fuse(x1, C1, x2, C2, out=None):
        x1, C1, x2, C2 = dev(x1), dev(C1), dev(x2), dev(C2)
        n, d = x1.t.shape
        xo, Co = out if out is not None else (DeviceArray(shape=(n, d)), DeviceArray(shape=(n, d, d)))
        check(lib().slb_datamodel_fuse(d, n, x1.ptr, C1.ptr, x2.ptr, C2.ptr, xo.ptr, Co.ptr, _stream()))
        return xo, Co

    @staticmethod
    def addsub(sign, x1, C1, x2, C2):
        x1, C1, x2, C2 = dev(x1), dev(C1), dev(x2), dev(C2)
        n, d = x1.t.shape
        xo, Co = DeviceArray(shape=(n, d)), DeviceArray(shape=(n, d, d))
        check(lib().slb_datamodel_addsub(d, n, sign, x1.ptr, C1.ptr, x2.ptr, C2.ptr, xo.ptr, Co.ptr, _stream()))
        return xo, Co

    @staticmethod
    def fuse_host(x1, C1, x2, C2):
        x1, C1, x2, C2 = _h(x1), _h(C1), _h(x2), _h(C2)
        n, d = x1.shape
        xo, Co = np.empty_like(x1), np.empty_like(C1)
        check(lib().slb_datamodel_fuse_host(d, n, _hp(x1), _hp(C1), _hp(x2), _hp(C2), _hp(xo), _hp(Co)))
        return xo, Co

    @staticmethod
    def safe_fuse(x1, C1, x2, C2, out=None):
        """DataModel<double,3>::safeFusion (DataModel.hpp:62-130), d = 3."""
        x1, C1, x2, C2 = dev(x1), dev(C1), dev(x2), dev(C2)
        n, d = x1.t.shape
        if d != 3:
            raise SlbError("safeFusion is only defined for d = 3 (DataModel.hpp:104)")
        xo, Co = out if out is not None else (DeviceArray(shape=(n, 3)), DeviceArray(shape=(n, 3, 3)))
        check(lib().slb_datamodel_safe_fuse(n, x1.ptr, C1.ptr, x2.ptr, C2.ptr, xo.ptr, Co.ptr, _stream()))
        return xo, Co


class ErrorStateEkf:
    """Batch of the error-state `Usckf` of src/filters/UsckfError.hpp (SURVEY 8f row f2): ekfPredict, ekfUpdate and
    ekfSingleUpdate with Joseph-form covariance updates, cloning.  State lives in device arrays laid out as the
    reference object holds it: mu (n x 48), err (n x 45), P (n x 45 x 45 dense)."""

    def __init__(self, mu, err, P):
        self.mu, self.err, self.P = dev(mu), dev(err), dev(P)
        self.n = self.mu.t.shape[0]
        torch = _torch()
        self.accepted = torch.zeros(self.n, dtype=torch.int32, device="cuda")

    def ekf_predict(self, F, Q):
        F, Q = dev(F), dev(Q)
        check(lib().slb_ekf_predict(self.n, self.err.ptr, self.P.ptr, F.ptr, Q.ptr, _stream()))

    def ekf_update(self, z, H, R, gate=True):
        z, H, R = dev(z), dev(H), dev(R)
        m = z.t.shape[1]
        ret = DeviceArray(shape=(self.n, m))
        check(lib().slb_ekf_update(self.n, m, self.mu.ptr, self.P.ptr, z.ptr, H.ptr, R.ptr, 1 if gate else 0, ret.ptr,
                                   C.c_void_p(self.accepted.data_ptr()), _stream()))
        return ret

    def ekf_single_update(self, z, H, R, gate=True):
        z, H, R = dev(z), dev(H), dev(R)
        m = z.t.shape[1]
        check(lib().slb_ekf_single_update(self.n, m, self.mu.ptr, self.err.ptr, self.P.ptr, z.ptr, H.ptr, R.ptr,
                                          1 if gate else 0, C.c_void_p(self.accepted.data_ptr()), _stream()))

    def cloning(self):
        check(lib().slb_ekf_clone(self.n, self.mu.ptr, self.err.ptr, self.P.ptr, _stream()))


class DeadReckon:
    """DeadReckon::updatePose with uncertainty and TransformWithUncertainty::operator* over n independent poses
    (DeadReckon.hpp:30-79,246-286; Transform.cpp:215-254).  Poses: pos(3) quat(w,x,y,z); covariances 6x6 over [r t]."""

    @staticmethod
    def compose(pose2, cov2, pose1, cov1):
        pose2, cov2, pose1, cov1 = dev(pose2), dev(cov2), dev(pose1), dev(cov1)
        n = pose2.t.shape[0]
        po, co = DeviceArray(shape=(n, 7)), DeviceArray(shape=(n, 6, 6))
        check(lib().slb_transform_compose(n, pose2.ptr, cov2.ptr, pose1.ptr, cov1.ptr, po.ptr, co.ptr, _stream()))
        return po, co

    @staticmethod
    def update_pose(dt, vel0, vel1, velcov, prev_pose, prev_cov, out=None):
        vel0, vel1, velcov, prev_pose, prev_cov = dev(vel0), dev(vel1), dev(velcov), dev(prev_pose), dev(prev_cov)
        n = vel0.t.shape[0]
        if out is None:
            out = (DeviceArray(shape=(n, 7)), DeviceArray(shape=(n, 6, 6)), DeviceArray(shape=(n, 7)), DeviceArray(shape=(n, 6, 6)))
        post, pcov, dpose, dcov = out
        check(lib().slb_deadreckon_update_pose(n, float(dt), vel0.ptr, vel1.ptr, velcov.ptr, prev_pose.ptr, prev_cov.ptr,
                                               post.ptr, pcov.ptr, dpose.ptr, dcov.ptr, _stream()))
        return post, pcov, dpose, dcov
