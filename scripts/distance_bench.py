#!/usr/bin/env python
"""Speed of the separation distance query (sffg_distance_poses_device) on the bench workload: building_s10 x
robot_small_s10, 2^24 device-resident Philox poses (bench.py's stream and range).  For each max_dist in {0.1 rho, rho,
4 rho, inf} (rho = the robot's bounding radius) it times `--launches` launches with CUDA events, alternating every launch
with one sffg_collide_poses_device launch on the same stream, and prints kernel ms and poses/s of both, the share of poses
in contact, capped, and measured, and the card it ran on.  GPU box only.

    python scripts/distance_bench.py [--launches 10] [--warmup 3] [--out profiles/distance_bench.json]
"""
import argparse
import json
import subprocess
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
import space_filling_forest_star_b200 as S  # noqa: E402

SEED = 0x5FF5EED
RANGE = [-70.0, 70.0, -70.0, 70.0, 0.0, 140.0]   # bench.py's pose range


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:   # (the numbers stand without it, but say so)
        return f"unknown ({e!r})"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--launches", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--poses", type=int, default=1 << 24)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    S.init(0)
    m = np.load(ROOT / "tests" / "golden" / "meshes.npz")
    obst, robot = m["building_s10"], m["robot_small_s10"]
    rho = float(np.linalg.norm(robot.reshape(-1, 3), axis=1).max())
    env = S.Environment(obst, robot)
    n = args.poses
    poses = S.gen_poses_device(SEED, 0, n, RANGE)
    dist = torch.empty(n, dtype=torch.float64, device="cuda")
    verdict = torch.empty(n, dtype=torch.uint8, device="cuda")

    def timed(fn):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        return a, b

    rows = []
    for label, md in (("0.1rho", 0.1 * rho), ("rho", rho), ("4rho", 4 * rho), ("inf", float("inf"))):
        for _ in range(args.warmup):
            env.distance_device(poses, md, out=dist)
            env.collide_device(poses, out=verdict)
        env.sync_check()
        ev_d, ev_c = [], []
        for _ in range(args.launches):
            ev_d.append(timed(lambda: env.distance_device(poses, md, out=dist)))
            ev_c.append(timed(lambda: env.collide_device(poses, out=verdict)))
        env.sync_check()
        td = [a.elapsed_time(b) for a, b in ev_d]
        tc = [a.elapsed_time(b) for a, b in ev_c]
        d = dist.cpu().numpy()
        v = verdict.cpu().numpy()
        assert np.array_equal(d == 0, v == 1), "distance 0 must be exactly the colliding poses"
        row = {"max_dist": label, "max_dist_value": md, "distance_ms": td, "collide_ms": tc,
               "distance_ms_median": float(np.median(td)), "collide_ms_median": float(np.median(tc)),
               "distance_poses_per_s": n / (np.median(td) * 1e-3), "collide_poses_per_s": n / (np.median(tc) * 1e-3),
               "contact_share": float((d == 0).mean()), "capped_share": float((d == md).mean()),
               "measured_share": float(((d > 0) & (d < md)).mean())}
        rows.append(row)
        print(f"max_dist {label:>6}: distance {row['distance_ms_median']:9.3f} ms ({row['distance_poses_per_s']:.3e} poses/s), "
              f"collide {row['collide_ms_median']:7.3f} ms; contact {row['contact_share']:.4f}, capped {row['capped_share']:.4f}, "
              f"measured {row['measured_share']:.4f}", flush=True)
    res = {"card": card(), "workload": "building_s10 x robot_small_s10, Philox poses in bench.py's range",
           "poses": n, "rho": rho, "launches": args.launches, "warmup": args.warmup, "rows": rows}
    print("card:", res["card"])
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
