#!/usr/bin/env python
"""Images/s of the GPD image projection: `prep.project` (crop + pgpd_gpd_project on the GPU, one call per cloud) and
the CPU dataset path (`projection.project_grasp`, one grasp per call with its own cKDTree, as a DataLoader worker
runs it), on a seeded view cloud of --points points (uniform in a 10 cm cube, like synth.make_tree) and grasps with
random poses inside it.  Prints one JSON line per configuration and writes them all to --out.

    python scripts/bench_project.py [--points 8000] [--grasps 64,1024,8192] [--chann 3,12] [--cpu-grasps 64] [--out F]

GPU times: CUDA events around --reps back-to-back calls after --warmup calls; each call includes the crop's host
synchronisation (prefix sum of the box counts).  The device name and power limit are read in the same run."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from pointnetgpd_b200 import prep, projection, synth  # noqa: E402
from pointnetgpd_b200.model.dataset import grasp_frame  # noqa: E402


def scene(P, G, seed=0):
    pc = synth.uniform(seed, (P, 3), -0.05, 0.05).astype(np.float32)
    g = np.zeros((G, 12))
    g[:, 0:3] = synth.uniform(seed + 1, (G, 3), -0.02, 0.02)
    g[:, 3:6] = synth.normal(seed + 2, (G, 3))
    g[:, 6] = 0.085
    g[:, 7] = synth.uniform(seed + 4, (G,), -np.pi, np.pi)
    return pc, g


def device_info():
    name = torch.cuda.get_device_name(0)
    try:
        power = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit", "--format=csv,noheader"],
                               capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        power = "unavailable"
    return name, power


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--points", type=int, default=8000)
    ap.add_argument("--grasps", default="64,1024,8192")
    ap.add_argument("--chann", default="3,12")
    ap.add_argument("--cpu-grasps", type=int, default=64)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_project.py measures the GPU path and needs a CUDA device")
    name, power = device_info()
    rows = []
    for chann in [int(c) for c in a.chann.split(",")]:
        for G in [int(g) for g in a.grasps.split(",")]:
            pc, grasps = scene(a.points, G)
            fr = prep.grasp_frames(grasps)
            pcd = torch.tensor(pc).cuda()
            for _ in range(a.warmup):
                img, valid = prep.project(pcd, fr, chann)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(a.reps):
                img, valid = prep.project(pcd, fr, chann)
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / a.reps
            offsets, _p, _i = prep.crop(pcd, fr)
            row = {"path": "gpu prep.project", "chann": chann, "points": a.points, "grasps": G, "ms_per_call": round(ms, 4),
                   "images_per_s": round(G / (ms * 1e-3), 1), "valid": int(valid.sum()),
                   "mean_in_box": round(float(offsets[-1]) / G, 1), "device": name, "power_limit": power}
            rows.append(row)
            print(json.dumps(row), flush=True)
        # the CPU dataset path on the first --cpu-grasps grasps of the same scene
        pc, grasps = scene(a.points, a.cpu_grasps)
        t0 = time.perf_counter()
        for g in range(a.cpu_grasps):
            center, rws, width = grasp_frame(grasps[g], np.eye(4))
            projection.project_grasp(pc, center, rws, width, chann)
        dt = time.perf_counter() - t0
        row = {"path": "cpu dataset (one process)", "chann": chann, "points": a.points, "grasps": a.cpu_grasps,
               "ms_per_image": round(dt * 1e3 / a.cpu_grasps, 3), "images_per_s": round(a.cpu_grasps / dt, 1),
               "cpu_threads": os.cpu_count(), "host_of": name}
        rows.append(row)
        print(json.dumps(row), flush=True)
    if a.out:
        with open(a.out, "w") as f:
            for r in rows:
                f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
