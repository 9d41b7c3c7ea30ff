#!/usr/bin/env python
"""Depth read from a CUDA array (orbit_depth_image, the form an imported Vulkan depth attachment takes) against depth read from
a linear buffer, on one GPU. Prints one JSON line.

  hiz_1080p / hiz_4k  orbit_hiz_build vs orbit_hiz_build_image (DepthPyramid.update with a tensor / a DepthImage)
  clusters_c4         orbit_light_cluster vs orbit_light_cluster_image (compute_clusters, C4 settings: 1920x1080, 120 px tiles,
                      24 slices)
  frame_c2            the C2 steady-state frame through PreparedFrame (main pass on, LATE + MAIN fused), depth from a tensor
                      (orbit_hiz_build_entity_cull_late) vs from a DepthImage (orbit_hiz_build_image_entity_cull_late)

Each arm is one CUDA graph per copy, replayed rotating over 3 copies of its inputs (depth buffer or array, pyramid, and for the
frame scene + camera state); us per call, median (and min) of --reps rounds. A parity bit per workload (the image arm's outputs
equal the linear arm's, byte for byte) is taken outside the timed region. `copy_pass_bytes` is what the image path saves the
integrator per camera and frame: an image-to-buffer copy of the depth (read + write), by arithmetic, not measured. The GPU name
and power limit are read in the same run.
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tools"), os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)
import numpy as np
import torch

from bench_views import gpu_identity, rotated_time
from orbit_b200 import frame, scenes
from orbit_b200.passes import ClusterSettings, Context, DepthPyramid, compute_clusters

N_COPIES = 3


def _u32(t):
    return t.cpu().numpy().view(np.uint32)


def _random_depth(w, h, seed):
    rng = np.random.default_rng(seed)
    d = rng.random((h, w), dtype=np.float32)
    d[rng.random((h, w)) < 0.3] = 0.0
    return d


def hiz(ctx, images, w, h, reps):
    depths = [torch.from_numpy(_random_depth(w, h, 17 + k)).to(ctx.device) for k in range(N_COPIES)]
    imgs = [images(d) for d in depths]
    lin = [DepthPyramid(ctx, "bdi_lin%d" % k, (w, h)) for k in range(N_COPIES)]
    tex = [DepthPyramid(ctx, "bdi_tex%d" % k, (w, h)) for k in range(N_COPIES)]
    for k in range(N_COPIES):
        lin[k].update(depths[k]); tex[k].update(imgs[k])
    torch.cuda.synchronize()
    same = all(np.array_equal(_u32(a.texels), _u32(b.texels)) for a, b in zip(lin, tex))
    t_lin = rotated_time([lambda k=k: lin[k].update(depths[k]) for k in range(N_COPIES)], reps)
    t_img = rotated_time([lambda k=k: tex[k].update(imgs[k]) for k in range(N_COPIES)], reps)
    return {"linear_us": t_lin, "image_us": t_img, "same_bytes": same, "copy_pass_bytes": 2 * 4 * w * h}


def clusters(ctx, images, scale, reps):
    sc, view = scenes.config_c4(scale)
    lights = scenes.make_lights(scenes.SEEDS["C4"], 65536 if scale >= 1.0 else 4096, sc.aabb_min, sc.aabb_max)
    ds = frame.DeviceScene.upload(ctx, sc, lights=lights)
    base = scenes.make_depth(sc, view)
    # three copies of the depth: the view's and two shifted by a few columns (same statistics, other bytes)
    depths = [torch.from_numpy(np.ascontiguousarray(np.roll(base, 3 * k, axis=1))).to(ctx.device) for k in range(N_COPIES)]
    imgs = [images(d) for d in depths]
    st = ClusterSettings(screen_resolution=(view.width, view.height), z_slice_count=24, tile_size_px=120)

    def run(src, k, tag):
        return compute_clusters(ctx, st, view.view, view.projection_matrix, view.near, src, ds.scene, name="bdi_cl_%s%d" % (tag, k))[0]
    keys = ("tile_depth_slice_mask", "cluster_depth_bounds", "unique_cluster_buffer", "light_offset_image", "light_index_buffer")
    same = True
    for k in range(N_COPIES):
        a, b = run(depths[k], k, "lin"), run(imgs[k], k, "img")
        torch.cuda.synchronize()
        same &= all(np.array_equal(getattr(a, x).cpu().numpy(), getattr(b, x).cpu().numpy()) for x in keys)
    t_lin = rotated_time([lambda k=k: run(depths[k], k, "lin") for k in range(N_COPIES)], reps)
    t_img = rotated_time([lambda k=k: run(imgs[k], k, "img") for k in range(N_COPIES)], reps)
    return {"linear_us": t_lin, "image_us": t_img, "same_bytes": bool(same), "lights": len(lights),
            "copy_pass_bytes": 2 * 4 * view.width * view.height}


def frame_c2(ctx, images, reps):
    import bench
    from test_gpu_hiz_entity_fused import _bytes
    sc, _ = scenes.config_c2()
    view = bench.c2_view(scenes, sc, 0)
    arms = {"linear": [], "image": []}
    for k in range(N_COPIES):
        ds = frame.DeviceScene.upload(ctx, sc)
        d = torch.from_numpy(scenes.make_depth(sc, view)).to(ctx.device)
        for arm, src in (("linear", d), ("image", images(d))):
            vs = frame.ViewState(ctx, ds, (view.width, view.height), name="bdi_%s%d" % (arm, k))
            pf = frame.PreparedFrame(ctx, ds, vs, view, src, name="bdi_%s%d" % (arm, k), main_pass=True)
            pf.launch(); pf.launch()
            arms[arm].append(pf)
    torch.cuda.synchronize()
    same = True
    for a, b in zip(arms["linear"], arms["image"]):
        x, y = _bytes(a), _bytes(b)
        same &= all(np.array_equal(x[key], y[key]) for key in x)
    out = {"same_bytes": bool(same), "copy_pass_bytes": 2 * 4 * view.width * view.height}
    for arm, pfs in arms.items():
        out[arm + "_us"] = rotated_time([pf.launch for pf in pfs], reps)
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--reps", type=int, default=21)
    ap.add_argument("--c4-scale", type=float, default=1.0, help="scenes.config_c4 scale of the cluster workload (1.0: 65536 lights)")
    ap.add_argument("--out", help="also write the JSON line to this file")
    args = ap.parse_args()
    from test_gpu_depth_image import Arrays, _image
    ctx = Context(0)
    arrays = Arrays(ctx.device)
    images = lambda d: _image(ctx, arrays, d)
    res = dict(gpu_identity(), reps=args.reps, copies=N_COPIES)
    res["hiz_1080p"] = hiz(ctx, images, 1920, 1080, args.reps)
    res["hiz_4k"] = hiz(ctx, images, 3840, 2160, args.reps)
    res["clusters_c4"] = clusters(ctx, images, args.c4_scale, args.reps)
    res["frame_c2"] = frame_c2(ctx, images, args.reps)
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")
    torch.cuda.synchronize()
    arrays.free()
    ctx.close()


if __name__ == "__main__":
    main()
