#!/usr/bin/env python
"""bench.py -- filter-steps/sec of the batched sigma-point filter hot path on N B200s of one node.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload ukfom|usckf|msckf|fusion|ekf|msckf_ekf|safefusion|deadreckon]
                  [--impl reference] [--dump-outputs DIR]

A "step" is one pass of the hot path (predict + update) over one batch of synthetic inputs.  The
default workload is BASELINE.json configs[3] (the north_star's): the Monte-Carlo USCKF fleet, 4M
instances over 8 GPUs = 524,288 per GPU (N = 48, m = 3), one fused predict+update launch per step.
The other GPU configs -- configs[1] batched UKFoM (65,536), configs[2] batched MSCKF (16,384),
configs[4] DataModel fusion (1M) -- are measured in the same run and nested under "also", each
with its own value / roofline / e2e.  One process per GPU (torchrun for N > 1); instances shard by
index with no collective on the step path ("weak" scaling: the per-GPU fleet is fixed); the only
NCCL traffic is the end-of-run all-reduce of the ensemble statistics, reported separately.

One JSON line is printed by rank 0; see the task contract for the keys.  `--impl reference` times
the reference's CPU algorithm instead: the dependency-free oracle port (the reference itself needs
Eigen/MTK/Boost, absent from this image) on all host cores, on a bounded sample of the same
workload.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from slam_localization_b200 import fleet, synth  # noqa: E402

L2_BYTES = 126 * 1024 * 1024
DUMP_BYTES = 60 * 10**6         # --dump-outputs: rows written at most; with the .npy headers the files stay under 64 MB


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


# ------------------------------------------------------------------------------------------------------
# clocks sampling during the timed region
# ------------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.monotonic(), line.strip()))

    def count(self, t0, t1):
        return sum(1 for (t, _) in self.rows if t0 <= t <= t1)

    def stop(self, t0=None, t1=None):
        """Summary of the samples that arrived in [t0, t1] (the loaded window); all samples if no window is given."""
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for (ts, r) in self.rows:
            if t0 is not None and not (t0 <= ts <= t1):
                continue
            f = [x.strip() for x in r.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                smax.append(float(f[2]))
            except ValueError:
                continue
            for n, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------------
# workloads
# ------------------------------------------------------------------------------------------------------
class UkfomWorkload:
    """BASELINE config 2: batched UKFoM (MTK9: pos, SO(3), vel), 65,536 instances per GPU, IMU predict +
    GPS update fused in one launch.  Several independent fleets are rotated so that consecutive
    steps never find their state in L2 (total resident footprint > 2x L2)."""
    name = "ukfom"
    metric = "filter-steps/sec (predict+update)"
    unit = "filter-steps/s"
    B = 65536
    layout = 9
    bytes_per_unit = 952            # SURVEY 8(d): 2*8*(45+10) + 72
    flops_per_unit = 1.4e4          # SURVEY 8(d)
    kernel = "slbd::ukf_kernel<MTK9, IMU, GPS, G=4, fused>"
    phases = ("ukf_kernel",)
    dominant = 0

    def __init__(self, rank, seed=1234):
        self.seed = seed + 1000 * rank
        self.sc = synth.ukfom_scenario(self.B, seed=self.seed, layout=self.layout, p_scale=1e-4)
        self.QD = 10

    def describe(self):
        return {"workload": "configs[1]: batched UKFoM, MTK9 pos/SO(3)/vel state, IMU predict + GPS update",
                "instances_per_gpu": self.B, "n": 9, "sigma_points": 19, "m": 3}

    def setup_gpu(self, engine, torch):
        per_fleet = (45 + 10) * 8 * self.B
        self.nfleets = max(2, int(np.ceil(2.2 * L2_BYTES / per_fleet)))
        self.fleets = []
        for _ in range(self.nfleets):
            f = engine.Ukf(self.B, layout=self.layout)
            f.set_state(self.sc["mu"], self.sc["P"])
            self.fleets.append(f)
        self.engine = engine
        self.Q = engine.DeviceArray(self.sc["Q"])
        self.R = engine.DeviceArray(self.sc["R"])
        self.u = [engine.DeviceArray(self.sc["u"]) for _ in range(2)]
        self.z = [engine.DeviceArray(self.sc["z"]) for _ in range(2)]
        # host (pinned) buffers for the end-to-end arm
        self.hu = torch.from_numpy(self.sc["u"].copy()).pin_memory()
        self.hz = torch.from_numpy(self.sc["z"].copy()).pin_memory()
        self.hQ = torch.from_numpy(self.sc["Q"].copy()).pin_memory()
        self.hR = torch.from_numpy(self.sc["R"].copy()).pin_memory()
        self.hmu = [torch.empty((self.B, self.QD), dtype=torch.float64).pin_memory() for _ in range(2)]
        self.l2_policy = "rotating %d resident fleets (%.0f MB > L2)" % (self.nfleets, self.nfleets * per_fleet / 1e6)

    def step(self, k):
        e = self.engine
        self.fleets[k % self.nfleets].step(e.PM_UKFOM_IMU, e.MM_GPS_POS, self.u[k & 1], self.sc["dt"], self.Q,
                                           self.z[k & 1], self.R)

    def step_e2e(self, k):
        e = self.engine
        self.fleets[k % self.nfleets].step_host(e.PM_UKFOM_IMU, e.MM_GPS_POS, self.hu, self.sc["dt"], self.hQ, self.hz,
                                                self.hR, mu_out=self.hmu[k & 1], wait=False)

    e2e_api = "slb_ukf_step_host_async per step (pinned host u/z in, posterior means out to one of two host buffers), slb_wait at the end"

    def e2e_drain(self):
        self.fleets[0].wait()

    def e2e_bytes(self):
        return (self.B * 9 + 81 + 9) * 8, self.B * self.QD * 8

    def units_per_step(self):
        return self.B

    def launches_per_step(self):
        return 1

    def status_ok(self):
        return all(sum(f.status_counts()) == 0 for f in self.fleets)

    def outputs(self, k):
        f = self.fleets[k % self.nfleets]
        return {"mu": f.mu(), "P": f.P(), "status": f.status()}

    def stats_tensor(self):
        return self.fleets[0].ensemble_stats().t

    def cpu_step(self, slo, nsample, nthreads):
        sc = self.sc
        t0 = time.perf_counter()
        slo.ukf_step(9, slo.PM_UKFOM_IMU, slo.MM_GPS_POS, sc["mu"][:nsample], sc["P"][:nsample], sc["u"][:nsample],
                     sc["dt"], sc["Q"], sc["z"][:nsample], sc["R"], nthreads=nthreads)
        return time.perf_counter() - t0


class FusionWorkload:
    """BASELINE config 5: DataModel covariance fusion, 1M 6-dof pairwise fusions per step."""
    name = "fusion"
    metric = "fusions/sec (DataModel::fusion, d=6)"
    unit = "fusions/s"
    B = 1 << 20
    d = 6
    bytes_per_unit = 648            # SURVEY 8(d): packed-symmetric accounting; dense traffic is 1008 B
    flops_per_unit = 2.6e3
    kernel = "slbd::datamodel_kernel<6, fusion>"
    phases = ("datamodel_kernel",)
    dominant = 0

    def __init__(self, rank, seed=99):
        self.sc = synth.fusion_scenario(self.B, d=self.d, seed=seed + rank)

    def describe(self):
        return {"workload": "configs[4]: DataModel covariance fusion, 6-dof, pairwise", "fusions_per_step": self.B}

    def setup_gpu(self, engine, torch):
        self.engine = engine
        self.a = [engine.DeviceArray(self.sc[k]) for k in ("x1", "C1", "x2", "C2")]
        self.out = (engine.DeviceArray(shape=(self.B, self.d)), engine.DeviceArray(shape=(self.B, self.d, self.d)))
        self.h = [torch.from_numpy(self.sc[k]).pin_memory() for k in ("x1", "C1", "x2", "C2")]
        self.ho = (torch.empty((self.B, self.d), dtype=torch.float64).pin_memory(),
                   torch.empty((self.B, self.d, self.d), dtype=torch.float64).pin_memory())
        self.l2_policy = "inputs+outputs 1057 MB per step > L2"

    def step(self, k):
        self.engine.DataModel.fuse(*self.a, out=self.out)

    def step_e2e(self, k):
        e = self.engine
        e.check(e.lib().slb_datamodel_fuse_host(self.d, self.B, *[e._ptr_of(t) for t in self.h],
                                                e._ptr_of(self.ho[0]), e._ptr_of(self.ho[1])))

    def e2e_bytes(self):
        return 2 * self.B * (self.d + self.d * self.d) * 8, self.B * (self.d + self.d * self.d) * 8

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
        slo.datamodel(0, sc["x1"][:nsample], sc["C1"][:nsample], sc["x2"][:nsample], sc["C2"][:nsample], nthreads=nthreads)
        return time.perf_counter() - t0


class UsckfWorkload:
    """BASELINE configs 1/4: Monte-Carlo USCKF fleet (n=12, N=36+3+9=48, m=3), 4M instances over 8 GPUs =
    524,288 per GPU, predict (IMU-style process model) + update (VO features) per step, ONE fused launch.
    The fleet is 2048 distinct seeded priors replicated on the device; inputs differ per instance."""
    name = "usckf"
    metric = "filter-steps/sec (predict+update)"
    unit = "filter-steps/s"
    B = 524288
    NPRIOR = 2048
    bytes_per_unit = 19704          # SURVEY 8(d): 2*8*(1176+51) + 72
    flops_per_unit = 1.5e5
    kernel = "slbd::usckf_step_kernel<PM_USCKF_TEST, 3, 9, predict+update fused>"

    def __init__(self, rank, seed=4321):
        self.sc = synth.usckf_scenario(self.NPRIOR, seed=seed + 1000 * rank)
        rng = np.random.default_rng(seed + 1000 * rank + 1)
        rep = self.B // self.NPRIOR
        self.u = np.concatenate([rng.normal(size=(self.B, 3)), rng.normal(size=(self.B, 3)) * 0.2], axis=1)
        self.z = np.tile(self.sc["mu"][:, 39:42], (rep, 1)) + rng.normal(size=(self.B, 3)) * 0.1

    def describe(self):
        return {"workload": "configs[3]/[0]: Monte-Carlo USCKF fleet, 12-dof state + 2 clones + 3+9 features (N=48), "
                            "IMU-style predict + 3-D VO update", "instances_per_gpu": self.B, "n": 12, "N": 48, "m": 3}

    def setup_gpu(self, engine, torch):
        self.engine = engine
        self.f = engine.Usckf(self.B, nk=3, nl=9)
        self.f.set_state(self.sc["mu"], self.sc["P"], replicate=True)
        self.Q = engine.DeviceArray(self.sc["Q"])
        self.R = engine.DeviceArray(self.sc["R"])
        self.du = engine.DeviceArray(self.u)
        self.dz = engine.DeviceArray(self.z)
        self.hu = torch.from_numpy(self.u).pin_memory()
        self.hz = torch.from_numpy(self.z).pin_memory()
        self.hQ = torch.from_numpy(self.sc["Q"].copy()).pin_memory()
        self.hR = torch.from_numpy(self.sc["R"].copy()).pin_memory()
        # the per-step readout is the current single state statek_i, what Usckf::muSingleState() returns by default
        # (Usckf.hpp:457-478): 13 of the 51 posterior scalars.  The whole augmented mean (muState(), :518) is timed too
        # and reported as e2e_full_posterior: 214 MB per step and GPU, which the host side of an 8-GPU box cannot absorb.
        self.hmu = [torch.empty((self.B, 13), dtype=torch.float64).pin_memory() for _ in range(2)]
        self.hmu_full = torch.empty((self.B, 51), dtype=torch.float64).pin_memory()
        self.l2_policy = "fleet state %.0f MB per step > L2" % (self.B * (1184 + 52) * 8 / 1e6)

    phases = ("usckf_step_kernel",)   # predict + update fused: the record crosses HBM once per step
    dominant = 0

    def step(self, k):
        e = self.engine
        self.f.step(e.PM_USCKF_TEST, e.MM_USCKF_VO, self.du, self.sc["dt"], self.Q, self.dz, self.R)

    def step_e2e(self, k):
        e = self.engine
        self.f.set_output_slice(26, 13)
        self.f.step_host(e.PM_USCKF_TEST, e.MM_USCKF_VO, self.hu, self.sc["dt"], self.hQ, self.hz, self.hR,
                         mu_out=self.hmu[k & 1], wait=False)

    def step_e2e_full(self, k):
        e = self.engine
        self.f.set_output_slice(0, 51)
        self.f.step_host(e.PM_USCKF_TEST, e.MM_USCKF_VO, self.hu, self.sc["dt"], self.hQ, self.hz, self.hR,
                         mu_out=self.hmu_full, wait=False)

    e2e_api = ("slb_usckf_step_host_async per step (pinned host u/z in; posterior statek_i = muSingleState() out to one of two "
               "host buffers), slb_wait at the end")

    def e2e_drain(self):
        self.f.wait()

    def e2e_bytes_full(self):
        return (self.B * 9 + 144 + 9) * 8, self.B * 51 * 8

    def e2e_bytes(self):
        return (self.B * 9 + 144 + 9) * 8, self.B * 13 * 8

    def units_per_step(self):
        return self.B

    def launches_per_step(self):
        return 1

    def status_ok(self):
        return sum(self.f.status_counts()) == 0

    def outputs(self, k):
        return {"mu": self.f.mu(), "P": self.f.P(), "status": self.f.status()}

    def stats_tensor(self):
        return self.f.ensemble_stats().t

    def cpu_step(self, slo, nsample, nthreads):
        # instance i of the fleet starts from prior i % NPRIOR with its own u / z: walk the sample in blocks of priors
        sc = self.sc
        t0 = time.perf_counter()
        for b0 in range(0, nsample, self.NPRIOR):
            n = min(self.NPRIOR, nsample - b0)
            slo.usckf_step(slo.PM_USCKF_TEST, slo.MM_USCKF_VO, 3, 9, sc["mu"][:n], sc["P"][:n], self.u[b0:b0 + n], sc["dt"],
                           sc["Q"], self.z[b0:b0 + n], sc["R"], nthreads=nthreads)
        return time.perf_counter() - t0


class MsckfWorkload:
    """BASELINE config 3: batched MSCKF, 10 stochastic clones (N = 72, 145 sigma points), 50 visual features per
    update (m = 100), 16,384 instances per GPU; predict (delta-pose model) + UKF-flavoured update with the
    per-feature chi-square gate, two launches.  512 distinct seeded priors are replicated on the device; the
    measurements differ per instance."""
    name = "msckf"
    metric = "filter-steps/sec (predict+update)"
    unit = "filter-steps/s"
    B = 16384
    NPRIOR = 512
    K = 10
    NFEAT = 50
    bytes_per_unit = 44176          # SURVEY 8(d): 2*8*(2628+83) + 800
    flops_per_unit = 1.3e7          # SURVEY 8(d)
    kernel = "slbd::msckf_update_kernel (+ predict12_kernel)"

    def __init__(self, rank, seed=777):
        self.sc = synth.msckf_scenario(self.NPRIOR, seed=seed + 1000 * rank, k=self.K, nfeat=self.NFEAT)
        rng = np.random.default_rng(seed + 1000 * rank + 1)
        rep = self.B // self.NPRIOR
        self.u = np.tile(self.sc["u"], (rep, 1))
        # zero-motion delta pose keeps the replayed fleet near its priors; pixel noise differs per instance
        self.u[:, 0:3] = 0.0
        self.u[:, 3:7] = [1.0, 0.0, 0.0, 0.0]
        self.z = np.tile(self.sc["z"], (rep, 1)) + rng.normal(size=(self.B, 2 * self.NFEAT)) * 1e-3

    def describe(self):
        return {"workload": "configs[2]: batched MSCKF, 10 stochastic clones (N=72), 50 visual features/update (m=100)",
                "instances_per_gpu": self.B, "N": 72, "sigma_points": 145, "m": 100}

    def setup_gpu(self, engine, torch):
        self.engine = engine
        self.f = engine.Msckf(self.B, nclones=self.K)
        self.f.set_state(self.sc["mu"], self.sc["P"], replicate=True)
        # a pristine copy of the fleet: the UKF update shrinks P every step, so each timed step starts from
        # the same priors (device-to-device restore outside the kernels being measured is NOT done: the
        # fleet simply keeps filtering; P stays SPD because predict adds Q every step)
        self.Q = engine.DeviceArray(self.sc["Q"])
        self.R = engine.DeviceArray(self.sc["R"])
        self.lm = engine.DeviceArray(self.sc["landmarks"])
        self.du = engine.DeviceArray(self.u)
        self.dz = engine.DeviceArray(self.z)
        self.hu = torch.from_numpy(self.u).pin_memory()
        self.hz = torch.from_numpy(self.z).pin_memory()
        self.hQ = torch.from_numpy(self.sc["Q"].copy()).pin_memory()
        self.hR = torch.from_numpy(self.sc["R"].copy()).pin_memory()
        self.hlm = torch.from_numpy(np.ascontiguousarray(self.sc["landmarks"])).pin_memory()
        self.hmu = torch.empty((self.B, 13 + 7 * self.K), dtype=torch.float64).pin_memory()
        self.l2_policy = "fleet state %.0f MB per step > L2" % (self.B * (2640 + 84) * 8 / 1e6)

    phases = ("predict12_kernel", "msckf_update_kernel")
    dominant = 1

    def step_phase(self, k, p):
        e = self.engine
        if p == 0:
            self.f.predict(e.PM_MSCKF_DELTAPOSE, self.du, 0.0, self.Q)
        else:
            self.f.update(e.MM_MSCKF_REPROJ, self.lm, self.dz, self.R)

    def step(self, k):
        self.step_phase(k, 0)
        self.step_phase(k, 1)

    def step_e2e(self, k):
        e = self.engine
        self.f.step_host(e.PM_MSCKF_DELTAPOSE, e.MM_MSCKF_REPROJ, self.hu, 0.0, self.hQ, self.hlm, self.hz, self.hR,
                         mu_out=self.hmu, wait=False)

    e2e_api = "slb_msckf_step_host_async per step (chunked H2D / kernels / D2H pipeline replayed as a CUDA graph), slb_wait at the end"

    def e2e_drain(self):
        self.f.wait()

    def e2e_bytes(self):
        return (self.B * (13 + 2 * self.NFEAT) + 144 + 3 * self.NFEAT + (2 * self.NFEAT) ** 2) * 8, self.B * (13 + 7 * self.K) * 8

    def units_per_step(self):
        return self.B

    def launches_per_step(self):
        return 2

    def status_ok(self):
        return sum(self.f.status_counts()) == 0

    def outputs(self, k):
        return {"mu": self.f.mu(), "P": self.f.P(), "status": self.f.status(), "outliers": self.f.outliers()}

    def stats_tensor(self):
        return self.f.ensemble_stats().t

    def cpu_step(self, slo, nsample, nthreads):
        sc = self.sc
        t0 = time.perf_counter()
        for b0 in range(0, nsample, self.NPRIOR):
            n = min(self.NPRIOR, nsample - b0)
            mu, P, _ = slo.msckf_predict(slo.PM_MSCKF_DELTAPOSE, self.K, sc["mu"][:n], sc["P"][:n], self.u[b0:b0 + n], 0.0,
                                         sc["Q"], nthreads=nthreads)
            slo.msckf_update(slo.MM_MSCKF_REPROJ, self.K, mu, P, sc["landmarks"], self.z[b0:b0 + n], sc["R"], nthreads=nthreads)
        return time.perf_counter() - t0


WORKLOADS = {"ukfom": UkfomWorkload, "fusion": FusionWorkload, "usckf": UsckfWorkload, "msckf": MsckfWorkload}


import bench_workloads  # noqa: E402  (SURVEY 8f "next" rows: ekf, safefusion, deadreckon)

for _cls in bench_workloads.WORKLOADS:
    WORKLOADS[_cls.name] = _cls


# ------------------------------------------------------------------------------------------------------
BOUND = {"usckf": "fp64", "ukfom": "fp64", "msckf": "fp64", "msckf_ekf": "fp64", "fusion": "hbm", "ekf": "hbm",
         "safefusion": "hbm", "deadreckon": "hbm"}   # BASELINE.md section 3: the binding roofline per config
ALSO = ("ukfom", "msckf", "fusion")                  # nested under "also" when the default workload runs


def config_of(wl, world):
    """The `config` object of the JSON line: identical in the b200 and the reference arm."""
    return dict(wl.describe(), l2="every step's state is larger than L2 or a rotating set of fleets is (see l2_policy)",
                parallelism="instance-index shard x%d, no step-path collective" % world)


def measured_traffic(name):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the workload's dominant kernel, from the committed
    ncu --set full capture of the same workload shape (profiles/traffic.json names the capture); None if absent."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        d = json.load(open(p)).get(name)
        return (float(d["bytes_per_launch"]), d["source"]) if d else (None, None)
    except Exception:
        return None, None


def cpu_baseline(wl, steps=3, warmup=1, budget_s=12.0):
    """Times the oracle (CPU restatement of the reference's algorithm) on all host threads over a
    bounded sample of the same workload, `steps` timed passes after `warmup`."""
    from oracle import slo
    slo.build()
    cores = slo.hardware_threads()
    n0 = min(wl.units_per_step(), 64 * cores)
    t = wl.cpu_step(slo, n0, cores)
    rate = n0 / t
    steps = max(1, steps)
    nsample = int(min(wl.units_per_step(), max(n0, rate * budget_s / (steps + warmup))))
    for _ in range(warmup):
        wl.cpu_step(slo, nsample, cores)
    ts = [wl.cpu_step(slo, nsample, cores) for _ in range(steps)]
    tot = sum(ts)
    return {"value": nsample * len(ts) / tot, "unit": wl.unit, "cores": cores, "kind": "port",
            "sample": "%d of %d units per step, %d step(s) after %d warm-up, oracle/libslo.so on %d threads" %
                      (nsample, wl.units_per_step(), len(ts), warmup, cores)}, tot / len(ts) * 1e3


def dump_outputs(wl, k, out_dir):
    """Writes what step k of the timed path left for its caller (wl.outputs(k): arrays with one row per instance) as
    out_dir/<name>.npy in float64, and out_dir/instance.npy with the instances the rows belong to: every instance when
    all fit in DUMP_BYTES, otherwise a sorted sample drawn with a fixed seed.  Two builds run with the same arguments
    see the same inputs, so their dumps compare array for array."""
    import torch
    arrays = wl.outputs(k)
    n = wl.units_per_step()
    assert all(a.shape[0] == n for a in arrays.values())
    per = 8 * (1 + sum(int(np.prod(a.shape[1:])) for a in arrays.values()))
    keep = min(n, DUMP_BYTES // per)
    idx = np.arange(n) if keep == n else np.sort(np.random.default_rng(0).choice(n, keep, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        a = a[torch.from_numpy(idx).to(a.device)].cpu().numpy() if isinstance(a, torch.Tensor) else a[idx]
        np.save(os.path.join(out_dir, name + ".npy"), a.astype(np.float64))
    np.save(os.path.join(out_dir, "instance.npy"), idx.astype(np.float64))


def run_reference(args, rank, world):
    if rank != 0:
        return 0
    wl = WORKLOADS[args.workload](0)
    cb, ms = cpu_baseline(wl, steps=max(3, args.steps), warmup=max(1, args.warmup), budget_s=60.0)
    line = {"impl": "reference", "metric": wl.metric, "value": cb["value"], "unit": wl.unit, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": config_of(wl, max(world, args.gpus)),
            "cpu_baseline": cb,
            "e2e": {"value": cb["value"], "unit": wl.unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "note": "reference's own Eigen/MTK code cannot be built in this image; timed arm is the oracle port"}
    print(json.dumps(line), flush=True)
    return 0


def measure(wl, args, ctx, sample_clocks, dump_dir=None):
    """Runs one workload's device-resident arm, end-to-end arm and stats gather; returns the result dict (rank 0)
    or None (other ranks).  ctx = (torch, dist, engine, rank, world, local).  With dump_dir, rank 0 writes the outputs
    of the last timed step there (dump_outputs)."""
    torch, dist, engine, rank, world, local = ctx

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def rank_max(x):
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    wl.setup_gpu(engine, torch)
    hbm_peak, peak_src = measured_peaks()

    # ---- device-resident arm -----------------------------------------------------------------------
    # the sampler starts before the warm-up so that nvidia-smi is already streaming (one line per 20 ms) when the timed
    # region begins; only lines that arrive while the GPU is under this workload's load are summarised
    sampler = ClockSampler(local)
    if rank == 0 and sample_clocks:
        sampler.start()
    for k in range(args.warmup):
        wl.step(k)
    barrier()
    n0 = engine.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    t_load0 = time.monotonic()
    e0.record()
    nph = len(wl.phases)
    mids = []
    if nph == 1:
        for k in range(args.steps):
            wl.step(args.warmup + k)
    else:  # an event after every launch but the last of a step: the dominant kernel's own duration
        for k in range(args.steps):
            row = []
            for p in range(nph):
                wl.step_phase(args.warmup + k, p)
                ev = torch.cuda.Event(enable_timing=True)
                ev.record()
                row.append(ev)
            mids.append(row)
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    if nph == 1:
        dom_ms = ms / args.steps
    else:
        tot = 0.0
        for k, row in enumerate(mids):
            start = (mids[k - 1][-1] if k else e0) if wl.dominant == 0 else row[wl.dominant - 1]
            tot += start.elapsed_time(row[wl.dominant])
        dom_ms = tot / args.steps
    launches = engine.launch_count() - n0
    t_load1 = time.monotonic()
    clocks = None
    if rank == 0 and sample_clocks:
        # a timed region shorter than a few sampling periods is followed by untimed steps of the same workload until at
        # least 5 samples were taken under load; they are not part of any reported time.  Not when the outputs of the
        # last timed step are to be written: those steps would move the state on.
        extended = False
        t_end = time.monotonic() + 1.0
        kx = args.warmup + args.steps
        while not dump_dir and sampler.proc and sampler.count(t_load0, t_load1) < 5 and time.monotonic() < t_end:
            for _ in range(8):
                wl.step(kx)
                kx += 1
            torch.cuda.synchronize()
            t_load1 = time.monotonic()
            extended = True
        clocks = sampler.stop(t_load0, t_load1)
        clocks["sampled_over"] = "timed region + untimed steps of the same workload" if extended else "timed region"
    if dump_dir and rank == 0:      # before the end-to-end arm below steps the workload again
        dump_outputs(wl, args.warmup + args.steps - 1, dump_dir)
    ms_max = rank_max(ms)
    units = wl.units_per_step() * args.steps * world
    value = units / (ms_max * 1e-3)
    ok = wl.status_ok()

    # ---- end-to-end arm: host buffers in, host result out, every step -------------------------------
    def time_e2e(step_fn, nbytes, ke):
        drain = getattr(wl, "e2e_drain", lambda: None)
        for k in range(3):
            step_fn(k)
        drain()
        barrier()
        t0 = time.perf_counter()
        e0.record()
        for k in range(ke):
            step_fn(k)
        drain()                     # pipelined host API: wait for the steps still in flight (inside the timed region)
        e1.record()
        barrier()
        wall = (time.perf_counter() - t0) * 1e3
        ms_e = rank_max(max(e0.elapsed_time(e1), wall))
        h2d, d2h = nbytes
        return {"value": wl.units_per_step() * ke * world / (ms_e * 1e-3), "unit": wl.unit,
                "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "steps": ke,
                "pcie_gbs_per_rank": (h2d + d2h) * ke / (ms_e * 1e-3) / 1e9}

    e2e, e2e_full = None, None
    if not args.no_e2e:
        ke = max(3, min(args.steps, 50))
        e2e = time_e2e(wl.step_e2e, wl.e2e_bytes(), ke)
        e2e["api"] = getattr(wl, "e2e_api", None)
        if hasattr(wl, "step_e2e_full"):
            e2e_full = time_e2e(wl.step_e2e_full, wl.e2e_bytes_full(), min(ke, 10))

    # ---- end-of-run ensemble statistics (the only collective; not on the step path) -----------------
    # slb_gather_stats: per-shard (count, sum x, sum x x^T) + ncclAllReduce inside the C library (its own communicator,
    # created through the C ABI; at N = 1 there is no communicator and the call is the local reduction alone)
    gather_ms, gather_count = None, None
    if wl.stats_tensor() is not None:
        comm = fleet.make_nccl_comm(engine, rank, world) if world > 1 else None
        fl = wl.fleets[0] if hasattr(wl, "fleets") else wl.f
        out = engine.DeviceArray(shape=(1 + fl.N + fl.N * fl.N,))
        fl.gather_stats(comm, out)          # warm-up (NCCL connects lazily)
        barrier()
        e0.record()
        fl.gather_stats(comm, out)
        e1.record()
        barrier()
        gather_ms = e0.elapsed_time(e1)
        gather_count = float(out.t[0].item())   # instances behind the merged statistics: world x fleet
        if comm is not None:
            comm.close()

    if rank != 0:
        return None
    ms_per_step = ms_max / args.steps
    launch_ms = dom_ms                # average duration of the dominant kernel's launches (CUDA events, rank 0)
    hbm_ach = wl.bytes_per_unit * wl.units_per_step() / (launch_ms * 1e-3) / 1e9
    fp64_peak = engine.fp64_peak_tflops()
    fp64_ach = wl.flops_per_unit * wl.units_per_step() / (ms_per_step * 1e-3) / 1e12
    traffic, traffic_src = measured_traffic(wl.name)
    common = {"traffic": traffic, "traffic_source": traffic_src, "kernel": wl.kernel, "kernel_ms": launch_ms,
              "launches_per_step": list(wl.phases)}
    r_hbm = dict({"bound": "hbm", "achieved": hbm_ach, "peak": hbm_peak, "unit": "GB/s", "frac": hbm_ach / hbm_peak,
                  "peak_source": peak_src, "algorithmic_bytes_per_unit": wl.bytes_per_unit}, **common)
    r_f64 = dict({"bound": "fp64", "achieved": fp64_ach, "peak": fp64_peak, "unit": "TFLOP/s",
                  "frac": fp64_ach / fp64_peak if fp64_peak else None,
                  "peak_source": "measured in this run (slb_bench_fp64_peak, register-resident DFMA; DMMA peak is the same)",
                  "algorithmic_flops_per_unit": wl.flops_per_unit, "over": "whole step (all launches)"}, **common)
    binding = BOUND.get(wl.name, "hbm")
    return {
        "metric": wl.metric, "value": value, "unit": wl.unit, "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": config_of(wl, world),
        "l2_policy": wl.l2_policy,
        "roofline": r_f64 if binding == "fp64" else r_hbm,       # the binding roofline (BASELINE.md section 3)
        "roofline_other": r_hbm if binding == "fp64" else r_f64,  # the non-binding one, for information
        "e2e": e2e, "e2e_full_posterior": e2e_full, "gpu_launches": launches, "clocks": clocks, "status_clean": ok,
        "ensemble_stats_allreduce_ms": gather_ms, "ensemble_stats_instances": gather_count,
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--workload", default="usckf", choices=sorted(WORKLOADS))
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-also", action="store_true", help="skip the nested runs of the other BASELINE configs")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step of the workload computed to DIR/<name>.npy (float64, <= 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl b200)")
    if args.warmup < 3 and args.impl == "b200":
        args.warmup = 3

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        return run_reference(args, rank, world)

    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        print(json.dumps({"error": "no CUDA device; the engine has no CPU fallback"}))
        return 2
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    from slam_localization_b200 import engine
    ctx = (torch, dist, engine, rank, world, local)

    wl = WORKLOADS[args.workload](rank)
    line = measure(wl, args, ctx, sample_clocks=True, dump_dir=args.dump_outputs)
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        line["cpu_baseline"], _ = cpu_baseline(wl)
    del wl
    import gc
    gc.collect()
    torch.cuda.empty_cache()

    # the other BASELINE configs, nested: one driver run covers configs[1..4]
    if args.workload == "usckf" and not args.no_also:
        also = {}
        for name in ALSO:
            w2 = WORKLOADS[name](rank)
            a2 = argparse.Namespace(**vars(args))
            if name == "ukfom":      # a 0.14 ms step: more steps so that the timed region is not dominated by jitter
                a2.steps = max(args.steps, 200)
            r = measure(w2, a2, ctx, sample_clocks=False)
            if rank == 0:
                keep = {k: r[k] for k in ("metric", "value", "unit", "steps", "ms_per_step", "config", "l2_policy", "roofline",
                                          "roofline_other", "e2e", "gpu_launches", "status_clean",
                                          "ensemble_stats_allreduce_ms", "ensemble_stats_instances")}
                if world == 1 and not args.no_cpu_baseline:
                    keep["cpu_baseline"], _ = cpu_baseline(w2, budget_s=5.0)
                also[name] = keep
            del w2
            gc.collect()
            torch.cuda.empty_cache()
        if rank == 0:
            line["also"] = also
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
