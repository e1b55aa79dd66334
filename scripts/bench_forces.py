#!/usr/bin/env python
"""bench_forces.py — cost of the wind (pies_b200_set_wind) on the flagship scene S3 (20 834 tet boxes in stacked columns,
1 000 032 boundary triangles, 562 518 nodes).

Writes one JSON object (to --out, and to stdout) with the card's name and power limit, read in the same run, and:
  tick        mean, spread and launches per tick (stats.msTick, CUDA events) of --ticks ticks in bench.py's contact
              window (after its 60 untimed ticks) of two identical solvers, ticked alternately, one of them with a
              light breeze from tick 60 on (max_abs_force reports its largest node force): weak enough to leave the
              contacts much as they were, so the difference is the cost of the wind rather than a different scene
  kernels     device time of k_wind_tri + k_force_gather per substep, from torch.profiler over --profile-ticks ticks
              with wind in a separate pass
  bytes       what the two kernels must move at least, from the scene's shapes: k_wind_tri reads 3 ids (12 B) and
              writes one float4 slot (16 B) per triangle and reads q and vel (32 B) per node; k_force_gather reads the
              CSR (4 B per node + 4 B per corner), every slot once (16 B per triangle) and writes fext (16 B per node);
              with the achieved bandwidth over that device time against the data-sheet 7.7 TB/s of one B200
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

PEAK_BYTES_PER_S = 7.7e12
WIND = dict(velocity=(1.0, 0.0, 0.5), normalDrag=0.01, tangentialDrag=0.01)


def gpu_info():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:   # the numbers are still worth printing, but say that the card is unknown
        return "unknown (%s)" % e


def make(bodies, preroll):
    import pies_b200 as pb
    from pies_b200 import scenes
    s = pb.Solver(**scenes.S3_OPTIONS)
    scenes.build_s3(s, bodies=bodies)
    for _ in range(preroll):
        s.tick()
    return s


def timed(solvers, ticks):
    rec = [([], []) for _ in solvers]
    for _ in range(ticks):
        for s, (ms, launches) in zip(solvers, rec):
            s.tick()
            st = s.stats()
            ms.append(st.msTick); launches.append(st.kernelLaunchesLastTick)
    for s in solvers:
        assert not s.simFailed
    return [dict(ms_per_tick=float(np.mean(ms)), ms_spread=float(np.max(ms) - np.min(ms)),
                 launches_per_tick=float(np.mean(launches))) for ms, launches in rec]


def min_bytes(n_nodes, n_tri):
    wind_tri = 12 * n_tri + 16 * n_tri + 32 * n_nodes
    gather = 4 * (n_nodes + 1) + 4 * 3 * n_tri + 16 * n_tri + 16 * n_nodes
    return wind_tri + gather


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--bodies", type=int, default=20834)
    ap.add_argument("--preroll", type=int, default=60, help="untimed ticks first (bench.py's contact window for S3)")
    ap.add_argument("--ticks", type=int, default=20)
    ap.add_argument("--profile-ticks", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r06a_bench_forces.json"))
    args = ap.parse_args()
    out = {"gpu": gpu_info(), "bodies": args.bodies, "wind": WIND}

    a, s = make(args.bodies, args.preroll), make(args.bodies, args.preroll)
    n_nodes, n_tri = len(s.positions), len(s.getTriangles())
    subs = s.getOptions().timeSubsteps
    out.update(nodes=n_nodes, triangles=n_tri, substeps_per_tick=subs)
    s.setWind(**WIND)
    no_wind, wind = timed([a, s], args.ticks)
    out["tick"] = {"no_wind": no_wind, "wind": wind}
    out["max_abs_force"] = float(np.abs(s.externalForces()).max())
    a.close(); s.close()

    import torch
    from torch.profiler import ProfilerActivity, profile
    s = make(args.bodies, args.preroll)
    s.setWind(**WIND)
    s.tick()   # first tick with wind: builds the node -> triangle CSR outside the profiled window
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(args.profile_ticks):
            s.tick()
    torch.cuda.synchronize()
    assert not s.simFailed
    s.close()
    k = {"k_wind_tri": [0.0, 0], "k_force_gather": [0.0, 0]}
    for e in prof.key_averages():
        t_us = getattr(e, "device_time_total", None)
        if t_us is None:
            t_us = e.cuda_time_total
        for name in k:
            if name in e.key:
                k[name][0] += t_us; k[name][1] += e.count
    substeps = args.profile_ticks * subs
    us = {name: v[0] / substeps for name, v in k.items()}
    total_us = sum(us.values())
    b = min_bytes(n_nodes, n_tri)
    out["kernels"] = dict(us_per_substep=us, launches={name: v[1] for name, v in k.items()}, substeps=substeps,
                          total_us_per_substep=total_us)
    out["bytes"] = dict(min_bytes_per_substep=b, achieved_bytes_per_s=b / (total_us * 1e-6) if total_us else None,
                        share_of_7_7_tb_s=(b / (total_us * 1e-6)) / PEAK_BYTES_PER_S if total_us else None)
    text = json.dumps(out)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(text + "\n")
    print(text)


if __name__ == "__main__":
    main()
