#!/usr/bin/env python
"""Batched views against the same views culled one at a time, on one GPU. Prints one JSON line.

Pass 0 (frame.cull_views: orbit_entity_cull_views + orbit_meshlet_cull_views against frame.cull_pass per view):
  C4  the four shadow cascades of scenes.cascade_views over the full 10 M-meshlet scene (latency-bound: short lists)
  C5  16 of the 256 cameras over the full 20 M-meshlet scene (640 MB of meshlets: inputs come from HBM, not L2)
Two-pass occlusion (--only c2x4): 4 C2 street cameras, EARLY -> Hi-Z -> LATE -> MAIN per camera, in the steady state, three ways:
  separate   frame.PreparedFrame per camera on one stream (LATE and MAIN unfused, 10 launches per camera; `separate_fused`:
             the fused LATE + MAIN form, 7 launches per camera)
  concurrent one context, stream and graph per camera, the four in flight together (bench.py's concurrent_views form)
  batched    frame.PreparedViews: orbit_*_cull_views_occlusion + orbit_hiz_build_views, 10 launches for the four cameras
  Each arm is one CUDA graph per multi-camera frame, replayed rotating over 3 copies of scene + camera state (inputs out of
  L2); us per 4-camera frame (median of --reps rounds). Parity bit: every camera's lists, bitmasks and pyramid from the
  batched arm equal the separate arm's, byte for byte.

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


def c2_view(scene, index):
    """Camera `index` of the C2 city: the street-level corner cameras of bench.py (index 0 = the named view)."""
    lo, hi = scene.aabb_min, scene.aabb_max
    corners = [(-6.0, -6.0, 30.0), (hi[0] + 2.0, -6.0, -30.0), (-6.0, hi[2] + 2.0, 150.0), (hi[0] + 2.0, hi[2] + 2.0, 210.0)]
    x, z, yaw = corners[index % 4]
    yaw = np.radians(yaw + 15.0 * (index // 4))
    return scenes.perspective_view((x, 2.0, z), (np.sin(yaw), 0.0, np.cos(yaw)), 1920, 1080)


def rotated_time(fns, reps, rounds=8):
    """us per call of fns[i](), each captured into its own CUDA graph and replayed rotating over i (median, min of reps)."""
    graphs = []
    for fn in fns:
        fn(); torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            fn()
        graphs.append(g)
    for g in graphs:
        g.replay()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for i in range(rounds * len(graphs)):
            graphs[i % len(graphs)].replay()
        b.record(); torch.cuda.synchronize()
        ts.append(a.elapsed_time(b) * 1e3 / (rounds * len(graphs)))
    return float(np.median(ts)), float(np.min(ts))


def two_pass_workload(ctx, scale, reps, n_cams=4, n_copies=3):
    sc, _ = scenes.config_c2(scale)
    views = [c2_view(sc, i) for i in range(n_cams)]
    depths = [scenes.make_depth(sc, v) for v in views]
    copies = []
    for i in range(n_copies):
        ds = frame.DeviceScene.upload(ctx, sc)
        dd = [torch.from_numpy(d).to(ctx.device) for d in depths]
        vs_sep = [frame.ViewState(ctx, ds, (v.width, v.height), name="tp%d_s%d" % (i, k)) for k, v in enumerate(views)]
        vs_bat = [frame.ViewState(ctx, ds, (v.width, v.height), name="tp%d_b%d" % (i, k)) for k, v in enumerate(views)]
        sep = [frame.PreparedFrame(ctx, ds, vs, v, d, name="tp%d_sep%d" % (i, k), main_pass=True, fuse_late_main=False)
               for k, (vs, v, d) in enumerate(zip(vs_sep, views, dd))]
        fused = [frame.PreparedFrame(ctx, ds, vs, v, d, name="tp%d_fus%d" % (i, k), main_pass=True)
                 for k, (vs, v, d) in enumerate(zip(vs_sep, views, dd))]
        bat = frame.PreparedViews(ctx, ds, vs_bat, views, dd, name="tp%d_bat" % i)
        copies.append({"ds": ds, "dd": dd, "vs_sep": vs_sep, "sep": sep, "fused": fused, "bat": bat, "vs_bat": vs_bat})
    res = {"cameras": n_cams, "meshlet_instances": int(sc.n_meshlet_instances), "scene_copies": n_copies}
    for c in copies:       # frames 0 and 1 from all-zero bits: the steady state, in both arms
        for _ in range(2):
            for pf in c["sep"]:
                pf.launch()
            c["bat"].launch()
    torch.cuda.synchronize()
    same = True
    for c in copies:
        for k, pf in enumerate(c["sep"]):
            ref = {"early": (pf.early_dispatch, pf.early_draws), "late": (pf.late_dispatch, pf.late_draws),
                   "main": (pf.main_dispatch, pf.main_draws)}
            got = c["bat"].outputs[k]
            same &= all(same_lists([got[s]], [ref[s]], pf.rcap, pf.dcap) for s in ref)
            for a, b in ((c["vs_bat"][k].entity_visibility, c["vs_sep"][k].entity_visibility),
                         (c["vs_bat"][k].meshlet_visibility, c["vs_sep"][k].meshlet_visibility),
                         (c["vs_bat"][k].depth_pyramid.texels, c["vs_sep"][k].depth_pyramid.texels)):
                same &= bool(torch.equal(a.view(torch.int32), b.view(torch.int32)))
    res["parity"] = same
    c0 = copies[0]
    res["draws_per_camera"] = {s: [int(c0["bat"].outputs[k][s][1][:4].cpu().numpy().view(np.uint32)[0]) for k in range(n_cams)]
                               for s in ("early", "late", "main")}
    arms = {"separate": lambda c: [pf.launch() for pf in c["sep"]], "separate_fused": lambda c: [pf.launch() for pf in c["fused"]],
            "batched": lambda c: c["bat"].launch()}
    for key, fn in arms.items():
        before = ctx.launch_count
        fn(c0); torch.cuda.synchronize()
        res[key + "_launches"] = ctx.launch_count - before
    for key, fn in arms.items():
        res[key + "_us"], res[key + "_us_min"] = rotated_time([lambda c=c, fn=fn: fn(c) for c in copies], reps)
    # concurrent: one context + stream + graph per camera, the cameras of a frame in flight together
    cv_ctx = [Context(0) for _ in range(n_cams)]
    cv_streams = [torch.cuda.Stream() for _ in range(n_cams)]
    cv = []
    for c in copies:
        row = []
        for k in range(n_cams):
            with torch.cuda.stream(cv_streams[k]):
                pf = frame.PreparedFrame(cv_ctx[k], c["ds"], c["vs_sep"][k], views[k], c["dd"][k], name="cv%d_%d" % (len(cv), k), main_pass=True)
                pf.launch(); pf.launch()
            torch.cuda.synchronize()
            pf.capture()
            row.append(pf)
        cv.append(row)
    torch.cuda.synchronize()

    def cv_run(rounds):
        main = torch.cuda.current_stream()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(main)
        for st in cv_streams:
            st.wait_event(a)
        for r in range(rounds * n_copies):
            for k in range(n_cams):
                with torch.cuda.stream(cv_streams[k]):
                    cv[r % n_copies][k].replay()
        for st in cv_streams:
            ev = torch.cuda.Event(); ev.record(st); main.wait_event(ev)
        b.record(main)
        torch.cuda.synchronize()
        return a.elapsed_time(b) * 1e3 / (rounds * n_copies)
    cv_run(2)
    ts = [cv_run(8) for _ in range(reps)]
    res["concurrent_us"], res["concurrent_us_min"] = float(np.median(ts)), float(np.min(ts))
    for key in ("separate", "separate_fused", "concurrent"):
        res["batched_speedup_vs_" + key] = res[key + "_us"] / res["batched_us"]
    for x in cv_ctx:
        x.close()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scale", type=float, default=1.0, help="scene scale (1.0 = the named configs)")
    ap.add_argument("--views", type=int, default=16, help="C5 cameras per batch (<= 16)")
    ap.add_argument("--reps", type=int, default=21)
    ap.add_argument("--only", choices=["c4", "c5", "c2x4"], default=None)
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
    if args.only in (None, "c2x4"):
        out["c2_four_cameras_two_pass"] = two_pass_workload(ctx, args.scale, args.reps)
    print(json.dumps(out), flush=True)
    ctx.close()


if __name__ == "__main__":
    main()
