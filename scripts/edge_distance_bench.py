#!/usr/bin/env python
"""Speed of the per-edge separation distance (sffg_distance_edges_device) on the bench environment: building_s10 x
robot_small_s10, length-4 edges from Philox starts (the edge batch of tests/test_gpu_fullsize.py), 2^20 edges at the
finite caps and 2^18 at max_dist = inf, both rotation modes.  For each cap it times `--launches` launches with CUDA events,
each followed on the same stream by one sffg_check_edges_device launch and by the do-it-yourself baseline: the same
samples expanded beforehand (not timed) through sffg_distance_poses_device, then a per-edge scatter_reduce minimum.
It counts the edges where the baseline and the edge call differ, and prints median kernel ms, the shares of edges in
contact, capped and measured, the host-call latency at m = 1, 64 and 1 024, and the card it ran on.  GPU box only.

    python scripts/edge_distance_bench.py [--launches 5] [--warmup 2] [--out profiles/edge_distance_bench.json]
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
import space_filling_forest_star_b200 as S  # noqa: E402
from distance_bench import card  # noqa: E402

SEED = 0x5FF5EED
START_RANGE = [-45.0, 45.0, -45.0, 45.0, 0.0, 125.0]
PI = 3.14159265358979323846


def edges(m, rot_mode):
    import torch
    s = S.gen_poses_device(SEED + 1, 0, m, START_RANGE).double()
    d = torch.randn((m, 3), device="cuda", dtype=torch.float64, generator=torch.Generator(device="cuda").manual_seed(1))
    e = s.clone()
    e[:, :3] += 4.0 * d / d.norm(dim=1, keepdim=True)
    if rot_mode == S.ROT_INTERPOLATE:
        e[:, 3:] = S.gen_poses_device(SEED + 2, 0, m, START_RANGE).double()[:, 3:]
    return s.contiguous(), e.contiguous()


def expand(s, e, rot_mode, sample=0.1):
    """the sample poses of every edge in the kernels' operation order, built with numpy on the host (torch's division by
    a scalar multiplies by the reciprocal, which moves samples by an ulp) -> (poses [N][6], edge of each pose), on the
    device"""
    import torch
    s, e = s.cpu().numpy(), e.cpu().numpy()
    wrap = lambda a: np.where(a < -PI, a + 2.0 * PI, np.where(a >= PI, a - 2.0 * PI, a))  # noqa: E731
    tot = np.zeros(len(s))
    for k in range(3):
        d = s[:, k] - e[:, k]
        tot = tot + d * d
    adir = wrap(e[:, 3:] - s[:, 3:])
    for k in range(3):
        tot = tot + adir[:, k] * adir[:, k]
    parts = np.sqrt(tot) / sample
    cnt = np.where(parts > 1.0, np.ceil(parts) - 1, 0).astype(np.int64)
    edge = np.repeat(np.arange(len(s)), cnt)
    idx = (np.arange(len(edge)) - np.repeat(np.cumsum(cnt) - cnt, cnt) + 1).astype(np.float64)
    p = np.zeros((len(edge), 6))
    pe = parts[edge]
    for k in range(3):
        p[:, k] = s[edge, k] + (idx * (e[edge, k] - s[edge, k])) / pe
        if rot_mode == S.ROT_INTERPOLATE:
            p[:, 3 + k] = s[edge, 3 + k] + (idx * adir[edge, k]) / pe
    return torch.from_numpy(p).cuda(), torch.from_numpy(edge).cuda()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--launches", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--edges", type=int, default=1 << 20)
    ap.add_argument("--edges-inf", type=int, default=1 << 18)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    S.init(0)
    m_ = np.load(ROOT / "tests" / "golden" / "meshes.npz")
    obst, robot = m_["building_s10"], m_["robot_small_s10"]
    rho = float(np.linalg.norm(robot.reshape(-1, 3), axis=1).max())
    env = S.Environment(obst, robot)

    def timed(fn):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        return a, b

    rows = []
    for rot_mode in (S.ROT_REFERENCE, S.ROT_INTERPOLATE):
        for label, md in (("0.1rho", 0.1 * rho), ("rho", rho), ("4rho", 4 * rho), ("inf", float("inf"))):
            m = args.edges_inf if label == "inf" else args.edges
            s, e = edges(m, rot_mode)
            poses, edge = expand(s, e, rot_mode)
            dist = torch.empty(m, dtype=torch.float64, device="cuda")
            free = torch.empty(m, dtype=torch.uint8, device="cuda")
            pdist = torch.empty(len(poses), dtype=torch.float64, device="cuda")
            base = torch.empty(m, dtype=torch.float64, device="cuda")

            def baseline():
                env.distance_device(poses, md, out=pdist)
                base.fill_(md)
                base.scatter_reduce_(0, edge, pdist, reduce="amin")

            for _ in range(args.warmup):
                env.edge_distance_device(s, e, md, rot_mode=rot_mode, out=dist)
                env.edges_device(s, e, 0.1, rot_mode, free_out=free)
                baseline()
            env.sync_check()
            ev_d, ev_c, ev_b = [], [], []
            for _ in range(args.launches):
                ev_d.append(timed(lambda: env.edge_distance_device(s, e, md, rot_mode=rot_mode, out=dist)))
                ev_c.append(timed(lambda: env.edges_device(s, e, 0.1, rot_mode, free_out=free)))
                ev_b.append(timed(baseline))
            env.sync_check()
            td, tc, tb = ([a.elapsed_time(b) for a, b in ev] for ev in (ev_d, ev_c, ev_b))
            d, f = dist.cpu().numpy(), free.cpu().numpy()
            assert np.array_equal(d == 0, f == 0), "distance 0 must be exactly the colliding edges"
            b = base.cpu().numpy()
            diff = d != b
            row = {"rot_mode": rot_mode, "max_dist": label, "max_dist_value": md, "edges": m, "samples": len(poses),
                   "edge_distance_ms": td, "check_edges_ms": tc, "baseline_ms": tb,
                   "edge_distance_ms_median": float(np.median(td)), "check_edges_ms_median": float(np.median(tc)),
                   "baseline_ms_median": float(np.median(tb)),
                   "edges_per_s": m / (np.median(td) * 1e-3),
                   "baseline_mismatch": int(diff.sum()), "baseline_lower": int((b < d).sum()),
                   "contact_share": float((d == 0).mean()), "capped_share": float((d == md).mean()),
                   "measured_share": float(((d > 0) & (d < md)).mean())}
            rows.append(row)
            print(f"mode {rot_mode} max_dist {label:>6} ({m} edges): edge distance {row['edge_distance_ms_median']:9.3f} ms, "
                  f"baseline {row['baseline_ms_median']:9.3f} ms, check_edges {row['check_edges_ms_median']:7.3f} ms; "
                  f"contact {row['contact_share']:.4f}, capped {row['capped_share']:.4f}, measured {row['measured_share']:.4f}; "
                  f"baseline differs on {row['baseline_mismatch']} edges",
                  flush=True)
            del poses, edge, pdist

    # host-call latency (planner-sized calls through the staging area), reference mode, max_dist = rho
    s, e = edges(1024, S.ROT_REFERENCE)
    hs, he = s.cpu().numpy(), e.cpu().numpy()
    lat = {}
    for m in (1, 64, 1024):
        for _ in range(5):
            env.EdgeDistance(hs[:m], he[:m], rho)
        t = []
        for _ in range(50):
            t0 = time.perf_counter()
            env.EdgeDistance(hs[:m], he[:m], rho)
            t.append((time.perf_counter() - t0) * 1e6)
        lat[str(m)] = {"median_us": float(np.median(t)), "min_us": float(np.min(t))}
        print(f"host call m={m}: median {lat[str(m)]['median_us']:.1f} us", flush=True)

    res = {"card": card(), "workload": "building_s10 x robot_small_s10, length-4 edges from Philox starts (seed + 1, "
           "range [-45,45]x[-45,45]x[0,125])", "rho": rho, "launches": args.launches, "warmup": args.warmup,
           "rows": rows, "host_latency_rho": lat}
    print("card:", res["card"])
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
