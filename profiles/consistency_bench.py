"""Cost of filter-consistency readout on the two sigma-point fleets.

Arms:
  step   a fused predict+update step timed with CUDA events over --steps steps after --warmup steps, NIS capture off vs
         on (slb_set_nis_capture), alternated --reps times in one process on two handles with the same prior and the
         same device-resident u / z: the default USCKF fleet (524 288 instances, nk = 3, nl = 9) and the UKFoM batch
         (65 536 instances, MTK9);
  nees   slb_consistency_stats with a truth and per-instance NEES output: the USCKF fleet's statek_i [24, 36) and its full
         48-dim state, the UKFoM batch's full 9-dim state; achieved GB/s against the algorithmic bytes below.
One JSON line per timed arm goes to stdout and to --out, with the card's name, power limit and SM clock.  Needs a CUDA
device (there is no CPU fallback).

    python profiles/consistency_bench.py --steps 200 --reps 3 --out profiles/r06_consistency_ab.jsonl
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader", "-i", "0"], capture_output=True,
                         text=True).stdout.strip()
    return dict(zip(q.split(","), [x.strip() for x in out.split(",")]))


def nees_bytes(n, qd, nis):
    """Algorithmic bytes per instance of one slb_consistency_stats call: the lower triangle of P_sub, the mean and truth
    scalars of the range (qd of each), the NEES written, the NIS read when capture is on."""
    return 8 * (n * (n + 1) // 2 + 2 * qd + 1 + (1 if nis else 0))


def setup(kind, engine, synth):
    if kind == "usckf":
        B, npri = 524288, 2048
        sc = synth.usckf_scenario(npri, seed=49)
        mk = lambda: engine.Usckf(B, nk=3, nl=9)                       # noqa: E731
        pm, mm = engine.PM_USCKF_TEST, engine.MM_USCKF_VO
        ranges = [("statek_i", 24, 12, 13), ("full", 0, 48, 51)]
    else:
        B, npri = 65536, 2048
        sc = synth.ukfom_scenario(npri, seed=31, layout=9)
        mk = lambda: engine.Ukf(B, layout=engine.LAYOUT_MTK9)           # noqa: E731
        pm, mm = engine.PM_UKFOM_IMU, engine.MM_GPS_POS
        ranges = [("full", 0, 9, 10)]
    rep = B // npri
    u = engine.DeviceArray(np.tile(sc["u"], (rep, 1)))
    z = engine.DeviceArray(np.tile(sc["z"], (rep, 1)))
    Q, R = engine.DeviceArray(sc["Q"]), engine.DeviceArray(sc["R"])
    arms = {}
    for arm in ("capture_off", "capture_on"):
        f = mk()
        f.set_state(sc["mu"], sc["P"], replicate=True)
        f.set_nis_capture(arm == "capture_on")
        arms[arm] = f
    truth = engine.DeviceArray(np.tile(sc["mu"], (rep, 1)) + 1e-3)
    step = lambda f: f.step(pm, mm, u, sc["dt"], Q, z, R)               # noqa: E731
    return B, arms, step, ranges, truth


def timed(torch, fn, steps, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--nees-calls", type=int, default=50)
    ap.add_argument("--workloads", default="usckf,ukfom")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("consistency_bench.py needs a CUDA device (no CPU fallback)")
    from slam_localization_b200 import engine, synth
    info = card()
    lines = []

    def emit(line):
        line["card"] = info
        print(json.dumps(line), flush=True)
        lines.append(line)
    for kind in args.workloads.split(","):
        B, arms, step, ranges, truth = setup(kind, engine, synth)
        for r in range(args.reps):
            for arm in ("capture_off", "capture_on"):
                f = arms[arm]
                ms = timed(torch, lambda: step(f), args.steps, args.warmup)
                emit(dict(workload=kind, arm=arm, run=r + 1, instances=B, steps=args.steps, ms_per_step=ms,
                          status_counts=f.status_counts()))
        f = arms["capture_on"]
        out, nees = engine.DeviceArray(shape=(6,)), engine.DeviceArray(shape=(B,))
        for name, t0, n, qd in ranges:
            call = lambda: engine.check(engine.lib().slb_consistency_stats(  # noqa: E731
                f.h, truth.ptr, t0, n, nees.ptr, out.ptr, engine._stream()))
            for r in range(args.reps):
                ms = timed(torch, call, args.nees_calls, 3)
                by = nees_bytes(n, qd, True) * B
                o = out.numpy()
                emit(dict(workload=kind, arm="nees_" + name, run=r + 1, instances=B, t0=t0, n=n, calls=args.nees_calls,
                          ms_per_call=ms, algorithmic_bytes=by, achieved_GBps=by / (ms * 1e-3) / 1e9,
                          nees_count=float(o[0]), anees=float(o[1] / max(o[0], 1)), nis_count=float(o[3])))
        del arms, f
        torch.cuda.empty_cache()
    for kind in args.workloads.split(","):
        for arm in sorted({x["arm"] for x in lines if x["workload"] == kind}):
            key = "ms_per_step" if arm.startswith("capture") else "ms_per_call"
            v = sorted(x[key] for x in lines if x["workload"] == kind and x["arm"] == arm)
            print("# %s %-14s median %.4f ms  spread %.4f ms (%d runs)" % (kind, arm, v[len(v) // 2], v[-1] - v[0], len(v)))
    if args.out:
        with open(args.out, "w") as fo:
            for x in lines:
                fo.write(json.dumps(x) + "\n")


if __name__ == "__main__":
    main()
