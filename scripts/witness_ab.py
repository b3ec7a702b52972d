#!/usr/bin/env python
"""A/B of the contact-witness probe on the bench workload (building_s10 x robot_small_s10, 2^24 Philox poses per launch):
one environment with the probe and one built with SFFG_WITNESS=0, timed alternately in rounds with CUDA events.  Prints
kernel ms and poses/s per round, warm build time and device memory of each environment, the traversal counters per pose
past the grid, whether both verdict buffers are byte-identical, and the card it ran on.  GPU box only.

    python scripts/witness_ab.py [--rounds 5] [--launches 10] [--out witness_ab.json]
"""
import argparse
import json
import os
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
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        return q
    except Exception as e:   # (the numbers stand without it, but say so)
        return f"unknown ({e!r})"


def make_env(obst, robot, witness):
    """the environment built twice, the second build's time is the warm one"""
    old = os.environ.get("SFFG_WITNESS")
    os.environ["SFFG_WITNESS"] = "1" if witness else "0"
    try:
        S.Environment(obst, robot).close()
        env = S.Environment(obst, robot)
    finally:
        if old is None:
            del os.environ["SFFG_WITNESS"]
        else:
            os.environ["SFFG_WITNESS"] = old
    return env


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--launches", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--poses", type=int, default=1 << 24)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    S.init(0)
    m = np.load(ROOT / "tests" / "golden" / "meshes.npz")
    obst, robot = m["building_s10"], m["robot_small_s10"]
    envs = {"probe_off": make_env(obst, robot, False), "probe_on": make_env(obst, robot, True)}
    P = args.poses
    poses = S.gen_poses_device(SEED, 0, P, RANGE)
    out = {k: torch.empty(P, dtype=torch.uint8, device="cuda") for k in envs}
    res = {"card": card(), "poses_per_launch": P, "rounds": args.rounds, "launches_per_round": args.launches, "arms": {}}
    for k, env in envs.items():
        info = env.info
        res["arms"][k] = {"build_ms_warm": info["build_ms"], "device_bytes": info["device_bytes"], "kernel_ms": []}
        for _ in range(args.warmup):
            env.collide_device(poses, out=out[k])
    torch.cuda.synchronize()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.launches)]
    for r in range(args.rounds):
        for k in (("probe_off", "probe_on") if r % 2 == 0 else ("probe_on", "probe_off")):
            env = envs[k]
            for a, b in ev:
                a.record()
                env.collide_device(poses, out=out[k])
                b.record()
            torch.cuda.synchronize()
            env.sync_check()
            ms = sum(a.elapsed_time(b) for a, b in ev) / len(ev)
            res["arms"][k]["kernel_ms"].append(ms)
            print(f"round {r} {k:9s} kernel {ms:.4f} ms  {P / (ms * 1e-3):.4g} poses/s", flush=True)
    res["verdicts_identical"] = bool(torch.equal(out["probe_on"], out["probe_off"]))
    res["collide_rate"] = float(out["probe_on"].float().mean().item())
    for k, env in envs.items():
        env.enable_counters(True)
        env.collide_device(poses, out=out[k])
        torch.cuda.synchronize()
        c = env.read_counters()
        env.enable_counters(False)
        g = max(c["poses_past_grid"], 1)
        a = res["arms"][k]
        a["counters"] = c
        a["per_pose_past_grid"] = {n: c[n] / g for n in ("traversal_steps", "box_tests", "triangles_transformed", "pair_tests",
                                                         "exact_run")}
        a["kernel_ms_min"], a["kernel_ms_max"] = min(a["kernel_ms"]), max(a["kernel_ms"])
        a["poses_per_s_best"] = P / (a["kernel_ms_min"] * 1e-3)
    on, off = res["arms"]["probe_on"], res["arms"]["probe_off"]
    res["kernel_gain"] = off["kernel_ms_min"] / on["kernel_ms_min"] - 1.0
    res["steps_ratio"] = on["per_pose_past_grid"]["traversal_steps"] / max(off["per_pose_past_grid"]["traversal_steps"], 1e-30)
    print(json.dumps(res, indent=1))
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
