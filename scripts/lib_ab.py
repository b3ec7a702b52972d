#!/usr/bin/env python
"""A/B of builds of the library on the pose kernel.  Each arm runs in a process of its own with SFFG_LIB naming its
build (the arm "default" is the in-tree library), and the arms alternate in every round.  Per arm and round: kernel ms per
launch of 2^24 float32 device poses on the bench stream (building_s10 x robot_small_s10, bench.py's seed and range, CUDA
events) and poses/s on cases T (triang_s10 x robot_cyl_small_s10) and D (dense3d_s1 x robot_small_s1), 2^22 poses each.
With --counters, once per arm: the work counters on the bench stream, the counters of the near-contact poses of
tests/test_gpu_clearance_planes.py (building_s10 walls and floors, float64 input), and a digest of every verdict buffer.
Prints the card and its power limit.  GPU box only.

    python scripts/lib_ab.py parent=path/to/libsffg_parent.so [other=...] [--rounds 3] [--counters] [--out ab.json]
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[1]
SEED = 0x5FF5EED
CASES = {   # (obstacles, robot, pose range, poses per launch); the bench workload is "B"
    "B": ("building_s10", "robot_small_s10", [-70.0, 70.0, -70.0, 70.0, 0.0, 140.0], 1 << 24),
    "T": ("triang_s10", "robot_cyl_small_s10", [-100.0, 100.0, -100.0, 100.0, 0.0, 100.0], 1 << 22),
    "D": ("dense3d_s1", "robot_small_s1", [-60.0, 2060.0, -60.0, 2110.0, 0.0, 1000.0], 1 << 22),
}


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:   # (the numbers stand without it, but say so)
        return f"unknown ({e!r})"


def near_contact_counters(S, meshes):
    """counters of the near-contact poses of test_near_contact_poses_at_the_walls (same seeds and offsets)"""
    sys.path.insert(0, str(ROOT / "tests"))
    import oracle as O
    from near_contact import boundary_brackets
    offsets, seed = (1e-2, 3e-3, 1e-3, 1e-4, 1e-5, 1e-6), SEED
    out = {}
    for rn in ("robot_small_s10", "robot_cyl_small_s10"):
        obst, rob = meshes["building_s10"], meshes[rn]
        env = S.Environment(obst, rob)
        for axis in (0, 2):
            lo, hi = boundary_brackets(O, O.ObbModel(obst), O.ObbModel(rob), seed + 7 + axis, 40000, CASES["B"][2], 0.5,
                                       axis=axis)
            poses = []
            for off in offsets:
                a, b = lo.copy(), hi.copy()
                a[:, axis] -= off
                b[:, axis] += off
                poses += [a, b]
            poses = np.concatenate(poses)
            env.enable_counters(True)
            v = env.Collide(poses)
            c = env.read_counters()
            env.enable_counters(False)
            out[f"{rn}_axis{axis}"] = {"poses": len(poses), "hit": float(v.mean()), "verdict_sha256": hashlib.sha256(v.tobytes()).hexdigest(),
                                       "counters": c}
        env.close()
    return out


def worker(args):
    sys.path.insert(0, str(ROOT))
    import torch
    import space_filling_forest_star_b200 as S
    S.init(0)
    meshes = np.load(ROOT / "tests" / "golden" / "meshes.npz")
    res = {"lib": str(S.lib_path()), "cases": {}}
    for key, (on, rn, rng, n) in CASES.items():
        env = S.Environment(meshes[on], meshes[rn])
        poses = S.gen_poses_device(SEED, 0, n, rng)
        out = torch.empty(n, dtype=torch.uint8, device="cuda")
        for _ in range(args.warmup):
            env.collide_device(poses, out=out)
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(args.launches):
            env.collide_device(poses, out=out)
        b.record()
        torch.cuda.synchronize()
        env.sync_check()
        ms = a.elapsed_time(b) / args.launches
        r = {"kernel_ms": ms, "poses_per_s": n / (ms * 1e-3)}
        if args.counters:
            r["verdict_sha256"] = hashlib.sha256(out.cpu().numpy().tobytes()).hexdigest()
            env.enable_counters(True)
            env.collide_device(poses, out=out)
            torch.cuda.synchronize()
            r["counters"] = env.read_counters()
            env.enable_counters(False)
        res["cases"][key] = r
        env.close()
    if args.counters:
        res["near_contact"] = near_contact_counters(S, meshes)
    print(json.dumps(res))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("arms", nargs="*", help="NAME=path/to/libsffg_x.so (the in-tree library is the arm 'default')")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--launches", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--counters", action="store_true")
    ap.add_argument("--worker", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if args.worker:
        worker(args)
        return
    arms = {"default": None}
    for a in args.arms:
        name, path = a.split("=", 1)
        arms[name] = str(Path(path).resolve())
    names = list(arms)
    res = {"card": card(), "rounds": args.rounds, "launches_per_round": args.launches,
           "poses_per_launch": {k: v[3] for k, v in CASES.items()}, "arms": {k: {"lib": v, "rounds": []} for k, v in arms.items()}}
    for r in range(args.rounds):
        order = names[r % len(names):] + names[:r % len(names)]
        for name in order:
            env = dict(os.environ)
            env.pop("SFFG_LIB", None)
            if arms[name]:
                env["SFFG_LIB"] = arms[name]
            cmd = [sys.executable, __file__, "--worker", "--launches", str(args.launches), "--warmup", str(args.warmup)]
            if args.counters and r == 0:
                cmd.append("--counters")
            p = subprocess.run(cmd, env=env, capture_output=True, text=True)
            if p.returncode != 0:
                sys.exit(f"arm {name} failed:\n{p.stdout[-2000:]}{p.stderr[-4000:]}")
            w = json.loads(p.stdout.strip().splitlines()[-1])
            res["arms"][name]["rounds"].append(w)
            print(f"round {r} {name:10s} " + "  ".join(f"{k} {c['kernel_ms']:.4f} ms {c['poses_per_s']:.4g}/s"
                                                       for k, c in w["cases"].items()), flush=True)
    for name, a in res["arms"].items():
        a["kernel_ms"] = {k: [w["cases"][k]["kernel_ms"] for w in a["rounds"]] for k in CASES}
        a["best_poses_per_s"] = {k: CASES[k][3] / (min(v) * 1e-3) for k, v in a["kernel_ms"].items()}
    print(json.dumps({k: {"kernel_ms": a["kernel_ms"], "best_poses_per_s": a["best_poses_per_s"]} for k, a in res["arms"].items()},
                     indent=1))
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
