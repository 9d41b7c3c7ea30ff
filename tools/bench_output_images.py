#!/usr/bin/env python
"""Outputs written into CUDA arrays (the depth pyramid mirrored into a mipmapped array, orbit_hiz_attach_image; the cluster
offset/count grid into a 3-D array, orbit_light_cluster_image_grid) against the linear outputs alone, on one GPU. Prints one
JSON line.

  hiz_1080p / hiz_4k   the Hi-Z build without and with a mirror, depth from a tensor (orbit_hiz_build) and from a DepthImage
                       (orbit_hiz_build_image)
  frame_c2             the C2 steady-state frame through PreparedFrame (main pass on, LATE + MAIN fused; depth from a tensor),
                       pyramid without and with a mirror (orbit_hiz_build_entity_cull_late with a mirror build)
  clusters_c4          compute_clusters from a DepthImage (C4 settings: 1920x1080, 120 px tiles, 24 slices) into a buffer
                       (orbit_light_cluster_image) and into a grid array (orbit_light_cluster_image_grid)

Each arm is one CUDA graph per copy, replayed rotating over 3 copies of its inputs and outputs; us per call, median (and min)
of --reps rounds. A parity bit per workload (the array equals the linear output, and the linear outputs equal the other arm's)
is taken outside the timed region. `mirror_bytes` / `grid_bytes` are the extra bytes the array arm stores. `copy_pass_bytes`
is what a separate buffer-to-image copy pass of the same output would move (read + write), by arithmetic, not measured. The GPU
name and power limit are read in the same run.
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
from orbit_b200.passes import ClusterGridImage, ClusterSettings, Context, DepthPyramid, compute_clusters

N_COPIES = 3


def _u32(t):
    return t.cpu().numpy().view(np.uint32)


def _random_depth(w, h, seed):
    rng = np.random.default_rng(seed)
    d = rng.random((h, w), dtype=np.float32)
    d[rng.random((h, w)) < 0.3] = 0.0
    return d


def _mirror_same(images, pyramid, mm):
    info = pyramid.info
    return all(np.array_equal(images.read_level(mm, l, max(info.width >> l, 1), max(info.height >> l, 1)), _u32(pyramid.level(l)))
               for l in range(info.levels))


def hiz(ctx, images, w, h, reps):
    from test_gpu_depth_image import _image
    depths = [torch.from_numpy(_random_depth(w, h, 17 + k)).to(ctx.device) for k in range(N_COPIES)]
    imgs = [_image(ctx, images, d) for d in depths]
    out = {}
    for form, srcs in (("tensor", depths), ("image", imgs)):
        plain = [DepthPyramid(ctx, "boi_plain%d" % k, (w, h)) for k in range(N_COPIES)]
        mms = [images.pyramid_array(plain[0].info) for _ in range(N_COPIES)]
        mirrored = [DepthPyramid(ctx, "boi_mirrored%d" % k, (w, h), image=mms[k]) for k in range(N_COPIES)]
        for k in range(N_COPIES):
            plain[k].update(srcs[k]); mirrored[k].update(srcs[k])
        torch.cuda.synchronize()
        same = all(np.array_equal(_u32(a.texels), _u32(b.texels)) and _mirror_same(images, b, mm) for a, b, mm in zip(plain, mirrored, mms))
        out[form] = {"plain_us": rotated_time([lambda k=k: plain[k].update(srcs[k]) for k in range(N_COPIES)], reps),
                     "mirror_us": rotated_time([lambda k=k: mirrored[k].update(srcs[k]) for k in range(N_COPIES)], reps),
                     "same_bytes": bool(same)}
    total = int(DepthPyramid(ctx, "boi_geometry", (w, h)).info.total_texels)
    out["mirror_bytes"] = 4 * total
    out["copy_pass_bytes"] = 2 * 4 * total
    return out


def frame_c2(ctx, images, reps):
    import bench
    from test_gpu_hiz_entity_fused import _bytes
    sc, _ = scenes.config_c2()
    view = bench.c2_view(scenes, sc, 0)
    arms = {"plain": [], "mirror": []}
    mms = []
    for k in range(N_COPIES):
        ds = frame.DeviceScene.upload(ctx, sc)
        d = torch.from_numpy(scenes.make_depth(sc, view)).to(ctx.device)
        for arm in arms:
            mm = None
            if arm == "mirror":
                mm = images.pyramid_array(DepthPyramid(ctx, "boi_geometry", (view.width, view.height)).info)
                mms.append(mm)
            vs = frame.ViewState(ctx, ds, (view.width, view.height), name="boi_%s%d" % (arm, k), pyramid_image=mm)
            pf = frame.PreparedFrame(ctx, ds, vs, view, d, name="boi_%s%d" % (arm, k), main_pass=True)
            pf.launch(); pf.launch()
            arms[arm].append(pf)
    torch.cuda.synchronize()
    same = True
    for a, b, mm in zip(arms["plain"], arms["mirror"], mms):
        x, y = _bytes(a), _bytes(b)
        same &= all(np.array_equal(x[key], y[key]) for key in x) and _mirror_same(images, b.vstate.depth_pyramid, mm)
    total = int(arms["plain"][0].vstate.depth_pyramid.info.total_texels)
    out = {"same_bytes": bool(same), "mirror_bytes": 4 * total, "copy_pass_bytes": 2 * 4 * total}
    for arm, pfs in arms.items():
        out[arm + "_us"] = rotated_time([pf.launch for pf in pfs], reps)
    return out


def clusters(ctx, images, scale, reps):
    from test_gpu_depth_image import _image
    sc, view = scenes.config_c4(scale)
    lights = scenes.make_lights(scenes.SEEDS["C4"], 65536 if scale >= 1.0 else 4096, sc.aabb_min, sc.aabb_max)
    ds = frame.DeviceScene.upload(ctx, sc, lights=lights)
    base = scenes.make_depth(sc, view)
    depths = [torch.from_numpy(np.ascontiguousarray(np.roll(base, 3 * k, axis=1))).to(ctx.device) for k in range(N_COPIES)]
    imgs = [_image(ctx, images, d) for d in depths]
    st = ClusterSettings(screen_resolution=(view.width, view.height), z_slice_count=24, tile_size_px=120)
    cx, cy, cz = st.cluster_counts()
    garrs = [images.grid(cx, cy, cz) for _ in range(N_COPIES)]
    grids = [ClusterGridImage(ctx, a) for a in garrs]

    def run(k, grid):
        return compute_clusters(ctx, st, view.view, view.projection_matrix, view.near, imgs[k], ds.scene,
                                name="boi_cl_%s%d" % ("grid" if grid else "buf", k), light_offset_image=grids[k] if grid else None)[0]
    keys = ("tile_depth_slice_mask", "cluster_depth_bounds", "unique_cluster_buffer", "light_index_buffer")
    same = True
    for k in range(N_COPIES):
        a, b = run(k, False), run(k, True)
        torch.cuda.synchronize()
        same &= all(np.array_equal(getattr(a, x).cpu().numpy(), getattr(b, x).cpu().numpy()) for x in keys)
        same &= np.array_equal(images.read_grid(garrs[k], cx, cy, cz), _u32(a.light_offset_image[:8 * cx * cy * cz]))
    n = cx * cy * cz
    return {"buffer_us": rotated_time([lambda k=k: run(k, False) for k in range(N_COPIES)], reps),
            "grid_us": rotated_time([lambda k=k: run(k, True) for k in range(N_COPIES)], reps),
            "same_bytes": bool(same), "lights": len(lights), "clusters": n, "grid_bytes": 8 * n, "copy_pass_bytes": 2 * 8 * n}


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--reps", type=int, default=21)
    ap.add_argument("--c4-scale", type=float, default=1.0, help="scenes.config_c4 scale of the cluster workload (1.0: 65536 lights)")
    ap.add_argument("--out", help="also write the JSON line to this file")
    args = ap.parse_args()
    from test_gpu_output_images import Images
    ctx = Context(0)
    images = Images(ctx.device)
    res = dict(gpu_identity(), reps=args.reps, copies=N_COPIES)
    res["hiz_1080p"] = hiz(ctx, images, 1920, 1080, args.reps)
    res["hiz_4k"] = hiz(ctx, images, 3840, 2160, args.reps)
    res["frame_c2"] = frame_c2(ctx, images, args.reps)
    res["clusters_c4"] = clusters(ctx, images, args.c4_scale, args.reps)
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")
    torch.cuda.synchronize()
    images.free()
    ctx.close()


if __name__ == "__main__":
    main()
