#!/usr/bin/env python
"""Speed of the continuous edge check (sffg_sweep_edges_device) on the bench environment: building_s10 x robot_small_s10,
length-4 edges from Philox starts (the batch of scripts/edge_distance_bench.py), 2^20 edges and a planner-sized 2 048,
both rotation modes, margin = 0.01 rho and 0.1 rho.  For each row it times `--launches` launches with CUDA events, each
followed on the same stream by one sffg_check_edges_device launch and by the do-it-yourself baseline: per edge, poses
expanded on the device at a tau spacing of at most margin / mu (not timed), sffg_distance_poses_device on them at
max_dist = 2 margin, a per-edge scatter_reduce minimum.  Every pose of the motion lies within margin / 2 of a grid pose in
distance, so a grid minimum >= margin is the same certificate (every pose >= margin / 2); the baseline decides the sweep's
answer where the minimum is >= 1.5 margin (every pose >= margin: clear) or < margin / 2 (some pose nearer: stopped), and
the script requires the two to agree there.  It records median kernel ms, the clear / stopped / contact shares, the host-call
latency at m = 1, 64 and 1 024, and the card.  GPU box only.

    python scripts/sweep_bench.py [--launches 5] [--warmup 2] [--out profiles/r03_sweep_bench.json]
"""
import argparse
import json
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "scripts"))
sys.path.insert(0, str(ROOT / "tests"))
import space_filling_forest_star_b200 as S  # noqa: E402
import sweep_motion as SM  # noqa: E402
from distance_bench import card  # noqa: E402
from edge_distance_bench import edges  # noqa: E402
from edge_samples import PI  # noqa: E402


def expand(s, e, rot_mode, margin, rho, chunk=1 << 16):
    """per edge ceil(mu / margin) + 1 evenly spaced taus on [0, 1], built on the device edge chunk by edge chunk (the taus
    need no particular rounding, only a spacing <= margin / mu) -> (poses [N][6], edge of each pose, taus per edge)"""
    import torch
    mu = SM.motion_bound(s.cpu().numpy(), e.cpu().numpy(), rho, rot_mode)
    cnt = torch.from_numpy(np.ceil(mu / margin).astype(np.int64) + 1).cuda()
    first = torch.cumsum(cnt, 0) - cnt
    total = int(cnt.sum())
    poses = torch.zeros((total, 6), dtype=torch.float64, device="cuda")
    edge = torch.repeat_interleave(torch.arange(len(s), device="cuda"), cnt)
    step = torch.zeros_like(s)
    step[:, :3] = e[:, :3] - s[:, :3]
    if rot_mode == S.ROT_INTERPOLATE:
        a = e[:, 3:] - s[:, 3:]
        step[:, 3:] = torch.where(a < -PI, a + 2.0 * PI, torch.where(a >= PI, a - 2.0 * PI, a))
    for lo in range(0, len(s), chunk):
        hi = min(lo + chunk, len(s))
        p0, p1 = int(first[lo]), int(first[hi - 1] + cnt[hi - 1])
        ed = edge[p0:p1]
        tau = ((torch.arange(p0, p1, device="cuda") - first[ed]).double() / (cnt[ed] - 1).clamp(min=1).double()).unsqueeze(1)
        poses[p0:p1] = s[ed] + tau * step[ed]
        if rot_mode != S.ROT_INTERPOLATE:
            poses[p0:p1, 3:] = 0.0
    return poses, edge, cnt.cpu().numpy()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--launches", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--edges", type=int, default=1 << 20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    S.init(0)
    m_ = np.load(ROOT / "tests" / "golden" / "meshes.npz")
    obst, robot = m_["building_s10"], m_["robot_small_s10"]
    rho = SM.radius(robot)
    env = S.Environment(obst, robot)

    def timed(fn):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        return a, b

    rows = []
    for rot_mode in (S.ROT_REFERENCE, S.ROT_INTERPOLATE):
        for m in (args.edges, 2048):
            for label, margin in (("0.01rho", 0.01 * rho), ("0.1rho", 0.1 * rho)):
                s, e = edges(m, rot_mode)
                poses, edge, cnt = expand(s, e, rot_mode, margin, rho)
                clear = torch.empty(m, dtype=torch.uint8, device="cuda")
                tt = torch.empty(m, dtype=torch.float64, device="cuda")
                dist = torch.empty(m, dtype=torch.float64, device="cuda")
                free = torch.empty(m, dtype=torch.uint8, device="cuda")
                pdist = torch.empty(len(poses), dtype=torch.float64, device="cuda")
                base = torch.empty(m, dtype=torch.float64, device="cuda")

                def sweep():
                    env.sweep_edges_device(s, e, margin, rot_mode, clear_out=clear, t_out=tt, dist_out=dist)

                def baseline():
                    env.distance_device(poses, 2 * margin, out=pdist)
                    base.fill_(2 * margin)
                    base.scatter_reduce_(0, edge, pdist, reduce="amin")

                for _ in range(args.warmup):
                    sweep()
                    env.edges_device(s, e, 0.1, rot_mode, free_out=free)
                    baseline()
                env.sync_check()
                ev_s, ev_c, ev_b = [], [], []
                for _ in range(args.launches):
                    ev_s.append(timed(sweep))
                    ev_c.append(timed(lambda: env.edges_device(s, e, 0.1, rot_mode, free_out=free)))
                    ev_b.append(timed(baseline))
                env.sync_check()
                ts, tc, tb = ([a.elapsed_time(b) for a, b in ev] for ev in (ev_s, ev_c, ev_b))
                c, d, b = clear.cpu().numpy(), dist.cpu().numpy(), base.cpu().numpy()
                f = free.cpu().numpy()
                # where the baseline decides the sweep's answer (allowing the pose query's 1e-9 S twice)
                tol = 2e-9 * max(1.0, float(np.abs(obst).max()), float(s[:, :3].abs().max()) + 4.0 + rho)
                b_clear, b_stop = b >= 1.5 * margin + tol, b < 0.5 * margin - tol
                disagree = int(((c == 1) & b_stop).sum() + ((c == 0) & b_clear).sum())
                assert disagree == 0, f"sweep and baseline disagree on {disagree} edges"
                assert np.all(f[c == 1] == 1), "a clear motion must pass isPathFree"
                row = {"rot_mode": rot_mode, "margin": label, "margin_value": margin, "edges": m,
                       "baseline_poses": len(poses), "baseline_poses_per_edge_mean": float(cnt.mean()),
                       "sweep_ms": ts, "check_edges_ms": tc, "baseline_ms": tb,
                       "sweep_ms_median": float(np.median(ts)), "check_edges_ms_median": float(np.median(tc)),
                       "baseline_ms_median": float(np.median(tb)), "edges_per_s": m / (np.median(ts) * 1e-3),
                       "baseline_decided": int((b_clear | b_stop).sum()), "baseline_disagree": disagree,
                       "baseline_certified": int((b >= margin).sum()),
                       "clear_share": float((c == 1).mean()), "stopped_share": float((c == 0).mean()),
                       "contact_share": float(((c == 0) & (d == 0)).mean()),
                       "isPathFree_free_share": float((f == 1).mean()),
                       "isPathFree_free_but_stopped": int(((f == 1) & (c == 0)).sum())}
                rows.append(row)
                print(f"mode {rot_mode} margin {label:>7} ({m} edges): sweep {row['sweep_ms_median']:9.3f} ms, baseline "
                      f"{row['baseline_ms_median']:9.3f} ms ({row['baseline_poses_per_edge_mean']:.0f} poses/edge), check_edges "
                      f"{row['check_edges_ms_median']:7.3f} ms; clear {row['clear_share']:.4f}, contact "
                      f"{row['contact_share']:.4f}; baseline decides {row['baseline_decided']}", flush=True)
                del poses, edge, pdist

    # host-call latency (planner-sized calls through the staging area), reference mode, margin = 0.1 rho
    s, e = edges(1024, S.ROT_REFERENCE)
    hs, he = s.cpu().numpy(), e.cpu().numpy()
    lat = {}
    for m in (1, 64, 1024):
        for _ in range(5):
            env.SweepEdges(hs[:m], he[:m], 0.1 * rho)
        t = []
        for _ in range(50):
            t0 = time.perf_counter()
            env.SweepEdges(hs[:m], he[:m], 0.1 * rho)
            t.append((time.perf_counter() - t0) * 1e6)
        lat[str(m)] = {"median_us": float(np.median(t)), "min_us": float(np.min(t))}
        print(f"host call m={m}: median {lat[str(m)]['median_us']:.1f} us", flush=True)

    res = {"card": card(), "workload": "building_s10 x robot_small_s10, length-4 edges from Philox starts (seed + 1, "
           "range [-45,45]x[-45,45]x[0,125])", "rho": rho, "launches": args.launches, "warmup": args.warmup,
           "rows": rows, "host_latency_0.1rho": lat}
    print("card:", res["card"])
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
