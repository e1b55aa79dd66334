#!/usr/bin/env python
"""bench_pick_drag.py — cost of picking (pies_b200_raycast) and dragging (pies_b200_set_drag_targets) on the flagship
scene S3 (20 834 tet boxes in stacked columns, 1 000 032 triangles).

Prints one JSON line with the card's name and power limit and:
  raycast     for 1, 64 and 1 024 rays aimed at random surface points of the built scene: CUDA-event time of the whole
              call (upload, the two kernels, the copy back; mean of --reps calls after one warm call) and ray-triangle
              tests per second (rays x triangles over that time)
  drag        for 0, 1 and 1 000 dragged nodes (targets 0.5 above their start, weight 1e3, reset every tick as an
              interactive host would): mean tick time (stats.msTick) and launches per tick over ticks 3..13 of a fresh
              solver (bench.py's free-fall window)
  drag_share  device time of k_drag_terms over the device time of all kernels with 1 000 drags, torch.profiler over
              --profile-ticks ticks of the free-fall window in a separate pass
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


def make(bodies):
    import pies_b200 as pb
    from pies_b200 import scenes
    s = pb.Solver(**scenes.S3_OPTIONS)
    scenes.build_s3(s, bodies=bodies)
    return s


def bench_raycast(s, args):
    import torch
    P = s.positions.astype(np.float64)
    tris = s.getTriangles().astype(np.int64)
    rng = np.random.default_rng(5)
    out = {}
    for n in (1, 64, 1024):
        f = rng.integers(0, len(tris), n)
        b = rng.dirichlet([1.0, 1.0, 1.0], n)
        tgt = b[:, :1] * P[tris[f, 0]] + b[:, 1:2] * P[tris[f, 1]] + b[:, 2:] * P[tris[f, 2]]
        o = tgt + np.array([0.0, 50.0, 0.0]) + rng.normal(size=(n, 3))
        d = (tgt - o).astype(np.float32)
        o = o.astype(np.float32)
        tri, _, _ = s.raycast(o, d)   # warm: loads the kernels, sizes the buffers
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(args.reps):
            s.raycast(o, d)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / args.reps
        out[str(n)] = dict(ms_per_call=ms, tests_per_s=n * len(tris) / (ms * 1e-3), hits=int((tri >= 0).sum()))
    out["triangles"] = int(len(tris))
    return out


def bench_drag(bodies, ndrag, profile_ticks):
    s = make(bodies)
    pos = s.positions
    ids = np.linspace(0, len(pos) - 1, ndrag).astype(np.uint32) if ndrag else np.zeros(0, np.uint32)
    tgt = pos[ids] + np.float32([0.0, 0.5, 0.0])
    w = np.full(len(ids), 1.0e3, np.float32)
    ms, launches = [], []
    for t in range(13):
        s.setDragTargets(ids, tgt, w)
        s.tick()
        if t >= 3:   # ticks 3..13
            st = s.stats()
            ms.append(st.msTick); launches.append(st.kernelLaunchesLastTick)
    share = None
    if profile_ticks and ndrag:
        s.close()
        s = make(bodies)
        for t in range(3):
            s.setDragTargets(ids, tgt, w); s.tick()
        import torch
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(profile_ticks):
                s.setDragTargets(ids, tgt, w); s.tick()
        tot = drag = 0.0
        for e in prof.key_averages():
            t_us = getattr(e, "device_time_total", None)
            if t_us is None:
                t_us = e.cuda_time_total
            if t_us <= 0:
                continue
            tot += t_us
            if "k_drag_terms" in e.key:
                drag += t_us
        share = drag / tot if tot else None
        torch.cuda.synchronize()
    assert not s.simFailed
    s.close()
    return dict(ms_per_tick=float(np.mean(ms)), ms_spread=float(np.max(ms) - np.min(ms)),
                launches_per_tick=float(np.mean(launches)), drag_share=share)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--bodies", type=int, default=20834)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--profile-ticks", type=int, default=5)
    args = ap.parse_args()
    out = {"gpu": gpu_info(), "bodies": args.bodies}
    s = make(args.bodies)
    out["raycast"] = bench_raycast(s, args)
    s.close()
    out["drag"] = {str(n): bench_drag(args.bodies, n, args.profile_ticks if n == 1000 else 0) for n in (0, 1, 1000)}
    print(json.dumps(out))


if __name__ == "__main__":
    main()
