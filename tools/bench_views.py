#!/usr/bin/env python
"""Batched pass-0 views (frame.cull_views: orbit_entity_cull_views + orbit_meshlet_cull_views) against the same views culled one
at a time (frame.cull_pass), on one GPU. Prints one JSON line.

  C4  the four shadow cascades of scenes.cascade_views over the full 10 M-meshlet scene (latency-bound: short lists)
  C5  16 of the 256 cameras over the full 20 M-meshlet scene (640 MB of meshlets: inputs come from HBM, not L2)

Times are CUDA-graph replays (median of --reps), as tools/bench_configs.py graph_time measures them. The launch counts of one
batch and a parity bit per workload (every view's buffers from the batched call == those of the separate calls, byte for
byte) are taken outside the timed region. The GPU name and power limit are read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
import numpy as np
import torch

from orbit_b200 import frame, scenes
from orbit_b200.passes import Context, OcclusionCullInfo


def graph_time(fn, reps):
    """us per call of fn(), captured once into a CUDA graph and replayed (median, min)."""
    fn(); torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        fn()
    g.replay(); torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); g.replay(); b.record(); torch.cuda.synchronize()
        ts.append(a.elapsed_time(b) * 1e3)
    return float(np.median(ts)), float(np.min(ts))


def gpu_identity():
    out = {"gpu": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        name, power = [x.strip() for x in q.split(",")]
        out.update(gpu=name, power_limit=power)
    except Exception as e:                     # the name from torch stays; say why the power limit is missing
        out["power_limit"] = "unavailable (%s)" % type(e).__name__
    return out


def same_lists(a, b, rcap, dcap):
    for x, y in zip(a, b):
        dx, dy = x[0].cpu().numpy(), y[0].cpu().numpy()
        n = int(dx[:4].view(np.uint32)[0])
        wx, wy = x[1].cpu().numpy(), y[1].cpu().numpy()
        m = int(wx[:4].view(np.uint32)[0])
        if not (np.array_equal(dx[:12 + 16 * min(n, rcap)], dy[:12 + 16 * min(n, rcap)]) and
                np.array_equal(wx[:4 + 28 * min(m, dcap)], wy[:4 + 28 * min(m, dcap)])):
            return False
    return True


def workload(ctx, name, sc, infos, reps):
    ds = frame.DeviceScene.upload(ctx, sc)
    rcap, dcap = int(ds.scene.record_capacity), int(ds.scene.draw_capacity)
    separate = lambda: [frame.cull_pass(ctx, "%s_sep%d" % (name, v), ds, ci) for v, ci in enumerate(infos)]
    batched = lambda: frame.cull_views(ctx, ds, infos, name=name + "_bat")
    res = {}
    for key, fn in (("separate", separate), ("batched", batched)):
        fn(); torch.cuda.synchronize()
        before = ctx.launch_count
        fn(); torch.cuda.synchronize()
        res[key + "_launches"] = ctx.launch_count - before
    res["separate_us"], res["separate_us_min"] = graph_time(separate, reps)
    res["batched_us"], res["batched_us_min"] = graph_time(batched, reps)
    a, b = separate(), batched()
    torch.cuda.synchronize()
    res["parity"] = same_lists(b, a, rcap, dcap)
    res["draws_per_view"] = [int(x[1][:4].cpu().numpy().view(np.uint32)[0]) for x in b]
    n = len(infos)
    res["views"] = n
    res["meshlet_instances"] = int(sc.n_meshlet_instances)
    for key in ("separate", "batched"):
        res[key + "_us_per_view"] = res[key + "_us"] / n
        res[key + "_gmeshlets_per_s"] = n * sc.n_meshlet_instances / res[key + "_us"] / 1e3
    res["speedup"] = res["separate_us"] / res["batched_us"]
    del ds
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scale", type=float, default=1.0, help="scene scale (1.0 = the named configs)")
    ap.add_argument("--views", type=int, default=16, help="C5 cameras per batch (<= 16)")
    ap.add_argument("--reps", type=int, default=21)
    ap.add_argument("--only", choices=["c4", "c5"], default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_views.py needs a CUDA device")
    ctx = Context(0)
    out = {"bench": "views", **gpu_identity(), "scale": args.scale, "reps": args.reps,
           "emit_ctas_per_sm_override": os.environ.get("ORBIT_EMIT_CTAS_PER_SM")}
    if args.only in (None, "c4"):
        sc, view = scenes.config_c4(args.scale)
        out["c4_cascades"] = workload(ctx, "c4", sc, [frame.cull_info_for(cv, OcclusionCullInfo("none")) for cv in scenes.cascade_views(view)],
                                      args.reps)
    if args.only in (None, "c5"):
        sc, views = scenes.config_c5(args.scale, n_views=256)
        out["c5_cameras"] = workload(ctx, "c5", sc, [frame.cull_info_for(v, OcclusionCullInfo("none")) for v in views[:args.views]], args.reps)
    print(json.dumps(out), flush=True)
    ctx.close()


if __name__ == "__main__":
    main()
