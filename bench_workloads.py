"""Bench workloads for the SURVEY 8(f) "next" rows (selected with bench.py --workload ekf|safefusion|deadreckon).
Same contract as the classes in bench.py: one step = one pass of the row's hot path over one synthetic batch;
outputs(k) returns what step k left for its caller, one row per instance."""
import time

import numpy as np

from slam_localization_b200 import synth


class EkfWorkload:
    """Row f2: error-state EKF of UsckfError.hpp, 3 x 15-DOF augmented state (N = 45), ekfPredict + Joseph-form
    ekfUpdate (delay-position measurement, m = 3) per step, two launches; every instance has its own F."""
    name = "ekf"
    metric = "filter-steps/sec (ekfPredict+ekfUpdate, Joseph form)"
    unit = "filter-steps/s"
    B = 262144
    NPRIOR = 4096
    # algorithmic bytes, packed-symmetric accounting like SURVEY 8(d): predict F 225 + r/w of P_ii (120), P_ik|P_il (450)
    # and mu_error_i (15); update r/w of the packed P (1035), mu 48, z 3, ret 3, accepted (4 B)
    bytes_per_unit = 8 * (225 + 2 * (120 + 450 + 15)) + 8 * (2 * 1035 + 48 + 3 + 3) + 4
    flops_per_unit = 2 * (15 * 45 * 15 + 15 * 15 * 15) + 2 * (45 * 45 * 3 + 1035 * 12)
    kernel = "slbd::ekf_update_kernel<3> (+ ekf_predict_kernel)"
    phases = ("ekf_predict_kernel", "ekf_update_kernel")
    dominant = 1

    def __init__(self, rank, seed=2024):
        self.sc = synth.ekf_scenario(self.NPRIOR, seed=seed + 1000 * rank)
        rep = self.B // self.NPRIOR
        rng = np.random.default_rng(seed + 1000 * rank + 1)
        self.F = np.eye(15)[None] + self.sc["dt"] * rng.normal(size=(self.B, 15, 15))
        self.z = np.tile(self.sc["z"], (rep, 1)) + 0.01 * rng.normal(size=(self.B, 3))
        self.rep = rep

    def describe(self):
        return {"workload": "SURVEY 8f row f2: error-state EKF (UsckfError.hpp), 3x15-dof augmented state (N=45), "
                            "ekfPredict + Joseph-form ekfUpdate (m=3)", "instances_per_gpu": self.B, "N": 45, "m": 3}

    def setup_gpu(self, engine, torch):
        self.engine, self.torch = engine, torch
        rep = self.rep
        mu = torch.from_numpy(self.sc["mu"]).cuda().repeat(rep, 1)
        err = torch.from_numpy(self.sc["err"]).cuda().repeat(rep, 1)
        P = torch.from_numpy(self.sc["P"]).cuda().repeat(rep, 1, 1)

        def wrap(t):
            a = engine.DeviceArray.__new__(engine.DeviceArray)
            a.t = t.contiguous()
            return a
        self.f = engine.ErrorStateEkf(wrap(mu), wrap(err), wrap(P))
        self.dF = engine.DeviceArray(self.F)
        self.dz = engine.DeviceArray(self.z)
        self.Q, self.H, self.R = (engine.DeviceArray(self.sc[k]) for k in ("Q", "H", "R"))
        self.hF = torch.from_numpy(self.F).pin_memory()
        self.hz = torch.from_numpy(self.z).pin_memory()
        self.hret = torch.empty((self.B, 3), dtype=torch.float64).pin_memory()
        self.hacc = torch.empty((self.B,), dtype=torch.int32).pin_memory()
        self.l2_policy = "fleet covariances %.0f MB per step > L2" % (self.B * 2025 * 8 / 1e6)

    def step_phase(self, k, p):
        if p == 0:
            self.f.ekf_predict(self.dF, self.Q)
        else:
            self.ret = self.f.ekf_update(self.dz, self.H, self.R, gate=False)

    def step(self, k):
        self.step_phase(k, 0)
        self.step_phase(k, 1)

    def step_e2e(self, k):
        # F (472 MB per step, the bulk of the input) is read by ekf_predict_kernel straight from the page-locked host
        # buffer (its LDGSTS record loads work unchanged on mapped memory); the small z goes through a copy
        self.dz.t.copy_(self.hz, non_blocking=True)
        self.f.ekf_predict(self.hF, self.Q)
        self.ret = self.f.ekf_update(self.dz, self.H, self.R, gate=False)
        self.hret.copy_(self.ret.t, non_blocking=True)
        self.hacc.copy_(self.f.accepted, non_blocking=True)
        self.torch.cuda.current_stream().synchronize()

    def e2e_bytes(self):
        return self.B * (225 + 3) * 8, self.B * (3 * 8 + 4)

    def units_per_step(self):
        return self.B

    def launches_per_step(self):
        return 2

    def status_ok(self):
        return bool(self.torch.isfinite(self.f.P.t[:: max(1, self.B // 64)]).all().item())

    def outputs(self, k):
        return {"err": self.f.err.t, "P": self.f.P.t, "ret": self.ret.t, "accepted": self.f.accepted}

    def stats_tensor(self):
        return None

    def cpu_step(self, slo, nsample, nthreads):
        sc = self.sc
        n = min(nsample, self.NPRIOR)
        t0 = time.perf_counter()
        err, P = slo.ekf_predict(sc["err"][:n], sc["P"][:n], self.F[:n], sc["Q"], nthreads=nthreads)
        slo.ekf_update(sc["mu"][:n], P, self.z[:n], sc["H"], sc["R"], gate=0, nthreads=nthreads)
        return (time.perf_counter() - t0) * nsample / n


class SafeFusionWorkload:
    """Row f3: DataModel<double,3>::safeFusion, 4M pairwise fusions per step."""
    name = "safefusion"
    metric = "fusions/sec (DataModel::safeFusion, d=3)"
    unit = "fusions/s"
    B = 1 << 22
    bytes_per_unit = 3 * 8 * (3 + 9)        # dense 3x3 in, in, out (the reference's storage)
    flops_per_unit = 900.0                  # 5 cofactor inverses, 2 Jacobi SVDs (~2 sweeps), 9 3x3 products
    kernel = "slbd::safe_fusion_kernel"
    phases = ("safe_fusion_kernel",)
    dominant = 0

    def __init__(self, rank, seed=5):
        self.sc = synth.safe_fusion_scenario(self.B, seed=seed + rank, log_spread=1.5)

    def describe(self):
        return {"workload": "SURVEY 8f row f3: DataModel::safeFusion, 3-dof, pairwise", "fusions_per_step": self.B}

    def setup_gpu(self, engine, torch):
        self.engine, self.torch = engine, torch
        self.a = [engine.DeviceArray(self.sc[k]) for k in ("x1", "C1", "x2", "C2")]
        self.out = (engine.DeviceArray(shape=(self.B, 3)), engine.DeviceArray(shape=(self.B, 3, 3)))
        self.h = [torch.from_numpy(self.sc[k]).pin_memory() for k in ("x1", "C1", "x2", "C2")]
        self.ho = (torch.empty((self.B, 3), dtype=torch.float64).pin_memory(),
                   torch.empty((self.B, 3, 3), dtype=torch.float64).pin_memory())
        self.l2_policy = "inputs+outputs %.0f MB per step > L2" % (self.B * 36 * 8 / 1e6)

    def step(self, k):
        self.engine.DataModel.safe_fuse(*self.a, out=self.out)

    def step_e2e(self, k):
        for d, h in zip(self.a, self.h):
            d.t.copy_(h, non_blocking=True)
        self.step(k)
        self.ho[0].copy_(self.out[0].t, non_blocking=True)
        self.ho[1].copy_(self.out[1].t, non_blocking=True)
        self.torch.cuda.current_stream().synchronize()

    def e2e_bytes(self):
        return 2 * self.B * 12 * 8, self.B * 12 * 8

    def units_per_step(self):
        return self.B

    def launches_per_step(self):
        return 1

    def status_ok(self):
        return True

    def outputs(self, k):
        return {"x": self.out[0].t, "C": self.out[1].t}

    def stats_tensor(self):
        return None

    def cpu_step(self, slo, nsample, nthreads):
        sc = self.sc
        t0 = time.perf_counter()
        slo.safe_fusion(sc["x1"][:nsample], sc["C1"][:nsample], sc["x2"][:nsample], sc["C2"][:nsample], nthreads=nthreads)
        return time.perf_counter() - t0


class DeadReckonWorkload:
    """Row f4: DeadReckon::updatePose with uncertainty (updateAttitude + TransformWithUncertainty::operator*),
    1M independent odometry streams per step; the posterior pose feeds the next step."""
    name = "deadreckon"
    metric = "pose-updates/sec (DeadReckon::updatePose with uncertainty)"
    unit = "pose-updates/s"
    B = 1 << 20
    bytes_per_unit = 8 * (12 + 2 * (7 + 36) + (7 + 36))   # vel0|vel1, prev pose+cov in, post pose+cov and delta pose+cov out
    flops_per_unit = 4.5e3
    kernel = "slbd::dr_update_pose_kernel"
    phases = ("dr_update_pose_kernel",)
    dominant = 0

    def __init__(self, rank, seed=11):
        self.sc = synth.deadreckon_scenario(self.B, seed=seed + rank)

    def describe(self):
        return {"workload": "SURVEY 8f row f4: DeadReckon::updatePose + TransformWithUncertainty composition",
                "poses_per_step": self.B}

    def setup_gpu(self, engine, torch):
        self.engine, self.torch = engine, torch
        sc = self.sc
        self.vel0, self.vel1, self.velcov = (engine.DeviceArray(sc[k]) for k in ("vel0", "vel1", "velcov"))
        self.pose = [engine.DeviceArray(sc["prev_pose"]), engine.DeviceArray(shape=(self.B, 7))]
        self.cov = [engine.DeviceArray(sc["prev_cov"]), engine.DeviceArray(shape=(self.B, 6, 6))]
        self.dpose, self.dcov = engine.DeviceArray(shape=(self.B, 7)), engine.DeviceArray(shape=(self.B, 6, 6))
        self.hv0 = torch.from_numpy(sc["vel0"]).pin_memory()
        self.hv1 = torch.from_numpy(sc["vel1"]).pin_memory()
        self.hpose = torch.empty((self.B, 7), dtype=torch.float64).pin_memory()
        self.hcov = torch.empty((self.B, 6, 6), dtype=torch.float64).pin_memory()
        self.l2_policy = "inputs+outputs %.0f MB per step > L2" % (self.B * self.bytes_per_unit / 1e6)
        self.k = 0

    def step(self, k):
        a, b = self.k & 1, (self.k + 1) & 1
        self.engine.DeadReckon.update_pose(self.sc["dt"], self.vel0, self.vel1, self.velcov, self.pose[a], self.cov[a],
                                           out=(self.pose[b], self.cov[b], self.dpose, self.dcov))
        self.k += 1

    def step_e2e(self, k):
        self.vel0.t.copy_(self.hv0, non_blocking=True)
        self.vel1.t.copy_(self.hv1, non_blocking=True)
        self.step(k)
        b = self.k & 1
        self.hpose.copy_(self.pose[b].t, non_blocking=True)
        self.hcov.copy_(self.cov[b].t, non_blocking=True)
        self.torch.cuda.current_stream().synchronize()

    def e2e_bytes(self):
        return self.B * 12 * 8, self.B * 43 * 8

    def units_per_step(self):
        return self.B

    def launches_per_step(self):
        return 1

    def status_ok(self):
        return bool(self.torch.isfinite(self.pose[self.k & 1].t[:: max(1, self.B // 64)]).all().item())

    def outputs(self, k):
        b = self.k & 1
        return {"pose": self.pose[b].t, "cov": self.cov[b].t, "delta_pose": self.dpose.t, "delta_cov": self.dcov.t}

    def stats_tensor(self):
        return None

    def cpu_step(self, slo, nsample, nthreads):
        sc = self.sc
        t0 = time.perf_counter()
        slo.dr_update_pose(sc["dt"], sc["vel0"][:nsample], sc["vel1"][:nsample], sc["velcov"], sc["prev_pose"][:nsample],
                           sc["prev_cov"][:nsample], nthreads=nthreads)
        return time.perf_counter() - t0


class MsckfEkfWorkload:
    """Row f1: batched MSCKF with the EKF-flavoured update (Jacobian, information-matrix outlier gate, QR compression),
    config-3 shapes: 10 clones (N = 72), 50 features (m = 100), 16,384 instances per GPU; predict + update, two launches."""
    name = "msckf_ekf"
    metric = "filter-steps/sec (predict + EKF update with QR compression)"
    unit = "filter-steps/s"
    B = 16384
    NPRIOR = 512
    K = 10
    NFEAT = 50
    bytes_per_unit = 44176          # same state traffic as the UKF flavour (SURVEY 8d): 2*8*(2628+83) + 800
    # information: H P H^T (sparse H) 0.13M + chol 100 0.33M + L^-1 0.33M; QR 100x72 0.79M + thin Q 0.79M;
    # Q^T R Q 2.5M; Hr P Hr^T 0.75M; chol 72 0.12M; TRSM 0.37M; Y Y^T 0.37M
    flops_per_unit = 6.5e6
    kernel = "slbd::msckf_ekf_update_kernel (+ predict12_kernel)"
    phases = ("predict12_kernel", "msckf_ekf_update_kernel")
    dominant = 1

    def __init__(self, rank, seed=777):
        self.sc = synth.msckf_scenario(self.NPRIOR, seed=seed + 1000 * rank, k=self.K, nfeat=self.NFEAT)
        rng = np.random.default_rng(seed + 1000 * rank + 1)
        rep = self.B // self.NPRIOR
        self.u = np.tile(self.sc["u"], (rep, 1))
        self.u[:, 0:3] = 0.0
        self.u[:, 3:7] = [1.0, 0.0, 0.0, 0.0]
        self.z = np.tile(self.sc["z"], (rep, 1)) + rng.normal(size=(self.B, 2 * self.NFEAT)) * 1e-3

    def describe(self):
        return {"workload": "SURVEY 8f row f1: batched MSCKF, EKF-flavoured update with outlier gate and QR compression, "
                            "10 clones (N=72), 50 features (m=100)", "instances_per_gpu": self.B, "N": 72, "m": 100}

    def setup_gpu(self, engine, torch):
        self.engine, self.torch = engine, torch
        self.f = engine.Msckf(self.B, nclones=self.K)
        self.f.set_state(self.sc["mu"], self.sc["P"], replicate=True)
        self.Q, self.R, self.lm = (engine.DeviceArray(self.sc[k]) for k in ("Q", "R", "landmarks"))
        self.du, self.dz = engine.DeviceArray(self.u), engine.DeviceArray(self.z)
        self.hu = torch.from_numpy(self.u).pin_memory()
        self.hz = torch.from_numpy(self.z).pin_memory()
        self.hmu = torch.empty((self.B, 13 + 7 * self.K), dtype=torch.float64).pin_memory()
        self.l2_policy = "fleet state %.0f MB per step > L2" % (self.B * (2640 + 84) * 8 / 1e6)

    def step_phase(self, k, p):
        e = self.engine
        if p == 0:
            self.f.predict(e.PM_MSCKF_DELTAPOSE, self.du, 0.0, self.Q)
        else:
            self.f.update_ekf(e.MM_MSCKF_REPROJ, self.lm, self.dz, self.R, gate=True)

    def step(self, k):
        self.step_phase(k, 0)
        self.step_phase(k, 1)

    def step_e2e(self, k):
        self.du.t.copy_(self.hu, non_blocking=True)
        self.dz.t.copy_(self.hz, non_blocking=True)
        self.step(k)
        self.hmu.copy_(self.torch.from_numpy(self.f.mu()))   # slb_download: device records -> host q-vectors

    def e2e_bytes(self):
        return self.B * (13 + 2 * self.NFEAT) * 8, self.B * (13 + 7 * self.K) * 8

    def units_per_step(self):
        return self.B

    def launches_per_step(self):
        return 2

    def status_ok(self):
        c = self.f.status_counts()   # gate rejections (bit 2) are expected; too few rows after the gate (QR_ROWS) is not
        return c[0] == 0 and c[1] == 0 and c[3] == 0 and c[4] == 0

    def outputs(self, k):
        return {"mu": self.f.mu(), "P": self.f.P(), "status": self.f.status(), "outliers": self.f.outliers()}

    def stats_tensor(self):
        return self.f.ensemble_stats().t

    def cpu_step(self, slo, nsample, nthreads):
        sc = self.sc
        n = min(nsample, self.NPRIOR)
        t0 = time.perf_counter()
        mu, P, _ = slo.msckf_predict(slo.PM_MSCKF_DELTAPOSE, self.K, sc["mu"][:n], sc["P"][:n], self.u[:n], 0.0, sc["Q"],
                                     nthreads=nthreads)
        slo.msckf_update_ekf(slo.MM_MSCKF_REPROJ, self.K, mu, P, sc["landmarks"], self.z[:n], sc["R"], nthreads=nthreads)
        return (time.perf_counter() - t0) * nsample / n


WORKLOADS = [EkfWorkload, SafeFusionWorkload, DeadReckonWorkload, MsckfEkfWorkload]
