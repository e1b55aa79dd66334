#!/usr/bin/env python
"""bench_colliders.py — cost of the static colliders on the flagship scene S3 (20 834 tet boxes in stacked columns).

Runs S3 twice in one process: as bench.py does (floor only) and inside a five-sided bin (four walls around the stack's
footprint, s3_translations extent plus --margin, and a bottom half-space at the floor).  Each run rolls forward untimed
to tick 65 and times the ticks of bench.py's window (65-85 with --steps 20 --warmup 5), then prints one JSON line:
  ms_per_tick        CUDA-event time of the tick (stats.msTick), mean over the window
  contacts_per_tick  node-collider contacts per tick (mask bits after each tick, read outside the tick's events)
  collider_share     device time of the collider kernels (k_collider_*, and the collider variant of k_tet_rhs /
                     k_gather_rhs_contacts counted whole) over the device time of all kernels, torch.profiler over
                     --profile-ticks extra ticks in a separate pass
plus the card's name and power limit.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:   # the numbers are still worth printing, but say that the card is unknown
        return "unknown (%s)" % e


def run(bodies, with_bin, args):
    import pies_b200 as pb
    from pies_b200 import scenes
    s = pb.Solver(**scenes.S3_OPTIONS)
    scenes.build_s3(s, bodies=bodies)
    cols = []
    if with_bin:
        pos = s.positions   # the footprint of the s3_translations columns, as built
        lo, hi = pos.min(0) - args.margin, pos.max(0) + args.margin
        cols = [pb.halfspace((lo[0], 0, 0), (1, 0, 0)), pb.halfspace((hi[0], 0, 0), (-1, 0, 0)),
                pb.halfspace((0, 0, lo[2]), (0, 0, 1)), pb.halfspace((0, 0, hi[2]), (0, 0, -1)),
                pb.halfspace((0, 0, 0), (0, 1, 0))]
        s.setColliders(cols)
    first = args.preroll + args.warmup
    for _ in range(first):
        s.tick()
    ms, contacts = [], []
    for _ in range(args.steps):
        s.tick()
        ms.append(s.stats().msTick)
        if with_bin:
            m = s.colliderContacts()
            contacts.append(int(sum(int(np.count_nonzero(m & (1 << k))) for k in range(len(cols)))))
    share = None
    if with_bin and args.profile_ticks:
        import torch
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(args.profile_ticks):
                s.tick()
        tot = col = 0.0
        for e in prof.key_averages():
            t_us = getattr(e, "device_time_total", None)
            if t_us is None:
                t_us = e.cuda_time_total
            if t_us <= 0:
                continue
            tot += t_us
            if "collider" in e.key or "ILb1E" in e.key:
                col += t_us
        share = col / tot if tot else None
        torch.cuda.synchronize()
    assert not s.simFailed
    s.close()
    return dict(ms_per_tick=float(np.mean(ms)), ms_spread=float(np.max(ms) - np.min(ms)),
                contacts_per_tick=float(np.mean(contacts)) if contacts else 0.0, collider_share=share)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--bodies", type=int, default=20834)
    ap.add_argument("--preroll", type=int, default=60)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--margin", type=float, default=0.5)
    ap.add_argument("--profile-ticks", type=int, default=3)
    args = ap.parse_args()
    out = {"gpu": gpu_info(), "bodies": args.bodies,
           "tick_window": [args.preroll + args.warmup, args.preroll + args.warmup + args.steps]}
    out["floor_only"] = run(args.bodies, False, args)
    out["bin"] = run(args.bodies, True, args)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
