"""Cost of per-instance process / measurement noise (slb_set_noise_layout) on the two sigma-point fleets.

Arms, each a fused predict+update step timed with CUDA events over --steps steps after --warmup steps:
  usckf  the default USCKF fleet (524 288 instances, nk = 3, nl = 9), shared Q / R  vs  a distinct Q (12 x 12) and
         R (3 x 3) per instance;
  ukfom  the UKFoM batch (65 536 instances, MTK9), the same way (Q 9 x 9, R 3 x 3).
The shared and per-instance arms alternate --reps times in one process, on two handles with the same prior and the
same device-resident u / z.  One JSON line per timed arm goes to stdout and to --out, with the card's name, power
limit and SM clock.  Needs a CUDA device (there is no CPU fallback).

    python profiles/noise_bench.py --steps 200 --reps 3 --out profiles/r05_per_instance_noise_ab.jsonl
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

# algorithmic bytes per instance and step: the record in and out, the inputs, and the noise entries the kernels read
# (lower triangles) when they are per instance
NOISE_BYTES = {"usckf": 8 * (78 + 6), "ukfom": 8 * (45 + 6)}
STORED_BYTES = {"usckf": 8 * (144 + 9), "ukfom": 8 * (81 + 9)}


def card():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader", "-i", "0"], capture_output=True,
                         text=True).stdout.strip()
    return dict(zip(q.split(","), [x.strip() for x in out.split(",")]))


def spd(rng, B, n, base):
    from slam_localization_b200 import synth
    return synth.random_spd(rng, B, n, 1.0, 10.0) * (base * 10.0 ** rng.uniform(-1, 1, size=(B, 1, 1)))


def setup(kind, torch, engine, synth):
    """Two handles with the same prior, the shared and the per-instance noise, device-resident inputs."""
    rng = np.random.default_rng(5)
    if kind == "usckf":
        B, npri = 524288, 2048
        sc = synth.usckf_scenario(npri, seed=49)
        mk = lambda: engine.Usckf(B, nk=3, nl=9)
        n, m, pm, mm = 12, 3, engine.PM_USCKF_TEST, engine.MM_USCKF_VO
    else:
        B, npri = 65536, 2048
        sc = synth.ukfom_scenario(npri, seed=31, layout=9)
        mk = lambda: engine.Ukf(B, layout=engine.LAYOUT_MTK9)
        n, m, pm, mm = 9, 3, engine.PM_UKFOM_IMU, engine.MM_GPS_POS
    rep = B // npri
    u = engine.DeviceArray(np.tile(sc["u"], (rep, 1)))
    z = engine.DeviceArray(np.tile(sc["z"], (rep, 1)))
    arms = {}
    for arm in ("shared", "per_instance"):
        f = mk()
        f.set_state(sc["mu"], sc["P"], replicate=True)
        if arm == "shared":
            Q, R = engine.DeviceArray(sc["Q"]), engine.DeviceArray(sc["R"])
        else:
            Q = engine.DeviceArray(spd(rng, B, n, float(np.abs(np.diag(sc["Q"])).mean())))
            R = engine.DeviceArray(spd(rng, B, m, float(sc["R"][0, 0])))
        arms[arm] = (f, Q, R)
    step = lambda f, Q, R: f.step(pm, mm, u, sc["dt"], Q, z, R)
    return B, arms, step


def time_arm(torch, f, Q, R, step, steps, warmup):
    for _ in range(warmup):
        step(f, Q, R)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        step(f, Q, R)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--workloads", default="usckf,ukfom")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("noise_bench.py needs a CUDA device (no CPU fallback)")
    from slam_localization_b200 import engine, synth
    info = card()
    lines = []
    for kind in args.workloads.split(","):
        B, arms, step = setup(kind, torch, engine, synth)
        for r in range(args.reps):
            for arm in ("shared", "per_instance"):
                f, Q, R = arms[arm]
                ms = time_arm(torch, f, Q, R, step, args.steps, args.warmup)
                st = f.status_counts()
                line = dict(workload=kind, arm=arm, run=r + 1, instances=B, steps=args.steps, ms_per_step=ms,
                            status_counts=st, noise_bytes_read_per_instance=NOISE_BYTES[kind] if arm != "shared" else 0,
                            noise_bytes_stored_per_instance=STORED_BYTES[kind] if arm != "shared" else 0, card=info)
                print(json.dumps(line), flush=True)
                lines.append(line)
        del arms
        torch.cuda.empty_cache()
    for kind in args.workloads.split(","):
        for arm in ("shared", "per_instance"):
            v = sorted(x["ms_per_step"] for x in lines if x["workload"] == kind and x["arm"] == arm)
            print("# %s %-12s median %.4f ms/step  spread %.4f ms (%d runs)" % (kind, arm, v[len(v) // 2], v[-1] - v[0], len(v)))
    if args.out:
        with open(args.out, "w") as fo:
            for x in lines:
                fo.write(json.dumps(x) + "\n")


if __name__ == "__main__":
    main()
