#!/usr/bin/env python
"""bench.py — headline benchmark of the B200 visibility pipeline (BASELINE.json metric: Gmeshlets culled/s).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

Workload (N=1): BASELINE config C2 — procedural 10k-entity / 2M-meshlet city, one 1920x1080 view, two-pass
occlusion. One *step* = the reference's culling of one steady-state frame (BASELINE.md protocol):
EARLY entity+meshlet cull (pass 1) -> Hi-Z build -> LATE entity+meshlet cull (pass 2) (forward.rs:266-403), then the
MAIN pass (pass 1 again with the bits the late pass wrote, forward.rs:518-548). LATE and MAIN run in their fused form
(orbit_entity_cull_late_main / orbit_meshlet_cull_late_main: the MAIN pass's tests repeat the LATE pass's, so one entity
kernel and one test kernel produce both passes' buffers, byte for byte): 7 kernel launches per step (entity_cull, meshlet
test + emit, hiz_build, entity_cull, meshlet test + one emit launch for the LATE and the MAIN list). `value` = scene meshlet instances x views / step time with every input resident in HBM;
the step rotates over 4 independent copies of the scene + view state (> L2) so inputs come from HBM.
Besides the contract's K timed steps the line carries `repeats` (5 x >= 50 steps: median and min), `moving_camera`
(a frame whose late pass finds survivors), and — nested, not separate lines — `c3_sharded` and `c5_many_view`:
the two BASELINE configs whose work is split over the ranks, each with a parity bit against the oracle.
N>1 (torchrun, one rank per GPU): views are sharded over GPUs with no data-path collective (each rank culls
its own instance of the C2 view on a replicated city) -> weak scaling; value = sum of meshlets over ranks / max-over-ranks time.

`e2e` = the same metric through the public pass API with HOST buffers: per step the frame-varying inputs
(entity transforms, entity draws, depth buffer) are copied from pinned host memory, the five stage calls run,
and the results (both draw-command lists with their counts) are read back to the host — all inside the timed region.
Static assets (meshlets, mesh infos, materials) stay resident like the reference's GpuAssets.

--impl reference: the reference's CPU implementation of the path = the oracle port (OpenMP, all host cores) on the
same config; rank 0 only.

--dump-outputs DIR: after the K timed steps, rank 0 writes what the last of them handed its caller as DIR/<name>.npy
(see step_outputs). The inputs are generated from fixed seeds, so two builds (or the two --impl arms) run with the same
arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402

METRIC = "Gmeshlets culled/s (C2: 10k entities / 2M meshlets, 1920x1080, two-pass occlusion, steady-state frame)"
UNIT = "Gmeshlets/s"
WORKLOAD = "C2 city 10k entities / 2M meshlets, one 1920x1080 view per GPU, steady-state frame: early cull + Hi-Z + late cull + main cull"
N_COPIES = 4
KERNELS_PER_STEP = 7    # early: entity_cull, meshlet test, meshlet_emit; hiz_build; late + main fused: entity_cull, meshlet test, one meshlet_emit launch for both lists
DUMP_LIMIT_BYTES = 64 * 2 ** 20


def c2_view(scenes, scene, index):
    """Camera `index` of the C2 city: street-level corner cameras looking into the city (index 0 = the named view)."""
    lo, hi = scene.aabb_min, scene.aabb_max
    corners = [(-6.0, -6.0, 30.0), (hi[0] + 2.0, -6.0, -30.0), (-6.0, hi[2] + 2.0, 150.0), (hi[0] + 2.0, hi[2] + 2.0, 210.0)]
    x, z, yaw = corners[index % 4]
    yaw = np.radians(yaw + 15.0 * (index // 4))
    return scenes.perspective_view((x, 2.0, z), (np.sin(yaw), 0.0, np.cos(yaw)), 1920, 1080)


class ClockSampler:
    FIELDS = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index):
        self.rows, self.proc, self.gpu = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.FIELDS,
                                          "--format=csv,noheader,nounits", "-lms", "20"], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm = [float(r[1]) for r in self.rows if len(r) >= 8 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 8 and r[2].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) >= 8:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def measured_peak_gbs():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_traffic_bytes():
    """dram__bytes_read.sum + dram__bytes_write.sum of the dominant kernel from the committed ncu --set full capture."""
    try:
        with open(os.path.join(ROOT, "profiles", "r2_meshlet_test_ncu.json")) as f:
            return int(json.load(f)["dram_traffic_bytes_per_launch"])
    except Exception:
        return None


def late_meshlet_algorithmic_bytes(records, n_draws, n_materials=16, passes_vis=2):
    """SURVEY §8(d) meshlet-stage formula, pass 2, WITHOUT the pyramid term (conservative: sampled texels are not
    counted): 32*L + 16*R + 12 + 64*E + 400 + 80*mats + 4*R (visibility read) + 4*R (visibility write) + 4 + 28*S."""
    lanes = int(records["meshlet_count"].sum())
    R = len(records)
    E = len(np.unique(records["entity_index"]))
    return 32 * lanes + 16 * R + 12 + 64 * E + 400 + 80 * n_materials + 4 * R * passes_vis + 4 + 28 * n_draws, lanes, R, E


def step_outputs(passes, entity_visibility, meshlet_visibility, hiz_texels):
    """What one step hands its caller: per pass ("early", "late", "main") the dispatch header, records, draw count and draw
    commands (`passes[k]` = (header, records, draws) as read_dispatch / read_draws return them), the two visibility bitmasks
    the next frame reads and the Hi-Z pyramid. 32-bit words become float64 (exact); the texels stay float32. A list with
    no entries (the late pass emits nothing in the steady state) is left out; its count and header say it is empty."""
    words = lambda a, cols: np.ascontiguousarray(a).view(np.uint32).reshape(-1, cols).astype(np.float64)
    out = {}
    for k, (hdr, recs, draws) in passes.items():
        out[k + "_dispatch_header"] = np.asarray(hdr, np.uint32).astype(np.float64)
        out[k + "_draw_count"] = np.array([len(draws)], np.float64)
        if len(recs):
            out[k + "_dispatch_records"] = words(recs, 4)
        if len(draws):
            out[k + "_draw_commands"] = words(draws, 7)
    out["entity_visibility"] = words(entity_visibility, 1).reshape(-1)
    out["meshlet_visibility"] = words(meshlet_visibility, 1).reshape(-1)
    out["hiz_texels"] = np.asarray(hiz_texels, np.float32).reshape(-1)
    return out


def dump_outputs(out_dir, arrays):
    # the dump is for comparing builds output for output, so it is refused rather than sampled (C2 dumps 16.5 MB)
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise RuntimeError("outputs of one step (%d bytes) exceed the %d-byte dump limit" % (total, DUMP_LIMIT_BYTES))
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


# ------------------------------------------------------------------------------------------------------------
def run_reference(args, rank, world):
    """Reference arm: the CPU restatement (oracle port, OpenMP) of the same step on the same config."""
    if rank != 0:
        return
    import oracle_ref as O
    from orbit_b200 import scenes
    O.build()
    O.lib().oracle_set_threads(os.cpu_count() or 1)     # torchrun exports OMP_NUM_THREADS=1: ask for every host thread explicitly
    scene, _ = scenes.config_c2()
    view = c2_view(scenes, scene, 0)
    depth = scenes.make_depth(scene, view)
    hs = O.HostScene(scene)

    def frame_once():
        out = O.depth_prepass_culling(hs, view, depth)
        out["main"] = O.main_pass_culling(hs, view)
        return out
    for _ in range(2):  # reach the steady state (frame 0 fills the visibility bits)
        frame_once()
    for _ in range(max(args.warmup, 1)):
        frame_once()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        out = frame_once()
    dt = (time.perf_counter() - t0) / args.steps
    if args.dump_outputs:
        passes = {k: O.parse_dispatch(out[k][0]) + (O.parse_draws(out[k][1])[1],) for k in ("early", "late", "main")}
        dump_outputs(args.dump_outputs, step_outputs(passes, hs.entity_visibility, hs.meshlet_visibility, hs.hiz_texels))
    value = scene.n_meshlet_instances / dt / 1e9
    cores = int(O.lib().oracle_threads())
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD,
                       "note": "the reference's GLSL needs Rust + a Vulkan loader (neither in the image); CPU restatement of the shaders (oracle port), one view"},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
                             "sample": "%d whole C2 frames (early + Hi-Z + late + main), OpenMP over %d host threads" % (args.steps, cores)},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)



def sha(a):
    import hashlib
    return hashlib.sha256(np.ascontiguousarray(a).view(np.uint8).tobytes()).hexdigest()[:16]


def event_us(fn, reps=5):
    import torch
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); fn(); b.record(); torch.cuda.synchronize()
        ts.append(a.elapsed_time(b) * 1e3)
    return float(np.median(ts)), float(np.min(ts))


def max_over_ranks(values, dev, world):
    import torch
    import torch.distributed as dist
    if world == 1:
        return [float(v) for v in values]
    t = torch.tensor(list(values), device=dev, dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return [float(v) for v in t.tolist()]


def moving_camera_extra(ctx, frame, scenes, scene, copies, O):
    """A frame whose late pass finds survivors: every scene copy alternates between the named C2 camera (A) and the same
    camera yawed by 15 degrees (B), both on ONE ViewState, so each frame reads the visibility bits the OTHER camera's
    frame wrote. Parity: copy 0's B-after-A frame against the oracle, outside the timed region."""
    import torch
    view_a, view_b = copies[0].view, c2_view(scenes, scene, 4)
    depth_b_np = scenes.make_depth(scene, view_b)
    pf_b = []
    for i, pf in enumerate(copies):
        d = torch.from_numpy(depth_b_np).to(ctx.device)
        q = frame.PreparedFrame(ctx, pf.dscene, pf.vstate, view_b, d, name="c%d_moved" % i, main_pass=True)
        q.launch(); pf.launch(); q.launch(); pf.launch()
        torch.cuda.synchronize()
        q.capture()
        pf_b.append(q)
    torch.cuda.synchronize()
    # parity: a FRESH view state (bits all zero) taken through frames A, A, B on the GPU and by the oracle alike (stale meshlet
    # words of entities rejected at the entity level make the bits depend on the whole history, so both sides follow the same one)
    ok = None
    if O is not None:
        vs2 = frame.ViewState(ctx, copies[0].dscene, (view_a.width, view_a.height), name="moved_parity")
        pa = frame.PreparedFrame(ctx, copies[0].dscene, vs2, view_a, copies[0].depth, name="parity_a", main_pass=True)
        pb = frame.PreparedFrame(ctx, copies[0].dscene, vs2, view_b, pf_b[0].depth, name="parity_b", main_pass=True)
        pa.launch(); pa.launch(); pb.launch()
        torch.cuda.synchronize()
        n_late_p, late_p = frame.read_draws(pb.late_draws)
        n_main_p, main_p = frame.read_draws(pb.main_draws)
        hs = O.HostScene(scene)
        depth_a_np = copies[0].depth.cpu().numpy()
        for v, d in [(view_a, depth_a_np)] * 2 + [(view_b, depth_b_np)]:
            o = O.depth_prepass_culling(hs, v, d)
            om = O.main_pass_culling(hs, v)
        on, od = O.parse_draws(o["late"][1]); mn, md = O.parse_draws(om[1])
        ok = bool(on == n_late_p and mn == n_main_p and on > 0 and sha(od) == sha(late_p) and sha(md) == sha(main_p))
    for pf, q in zip(copies, pf_b):
        pf.launch(); pf.launch(); q.launch()
    torch.cuda.synchronize()
    n_late_b, _ = frame.read_draws(pf_b[0].late_draws, capacity=0)
    n_main_b, _ = frame.read_draws(pf_b[0].main_draws, capacity=0)
    copies[0].launch()
    torch.cuda.synchronize()
    n_late_a, _ = frame.read_draws(copies[0].late_draws, capacity=0)
    # timed: A on every copy, then B on every copy, ... (a copy's two frames are separated by the other copies' frames: inputs out of L2)
    def sweep(rounds):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(rounds):
            for q in pf_b:
                q.replay()
            for pf in copies:
                pf.replay()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / (rounds * 2 * len(copies))
    sweep(2)
    ms = [sweep(8) for _ in range(5)]
    for pf in copies:      # back to camera A's steady state for whatever follows
        pf.launch(); pf.launch()
    torch.cuda.synchronize()
    return {"what": "camera alternates between the named view and the same view yawed by 15 degrees: every frame reads the other camera's visibility bits, so the late pass tests AND emits",
            "ms_per_step_median": float(np.median(ms)), "ms_per_step_min": float(np.min(ms)),
            "late_survivors": [int(n_late_b), int(n_late_a)], "main_survivors_moved": int(n_main_b),
            "value": scene.n_meshlet_instances / (float(np.median(ms)) * 1e-3) / 1e9, "unit": UNIT, "bit_exact_vs_oracle": ok}


def c3_sharded_extra(ctx, rank, world, O):
    """BASELINE config C3: one 3840x2160 view over 50 M instanced meshlets, entity ranges split over the ranks (equal
    meshlet sums), depth pyramid distributed, survivor lists gathered on rank 0 (the GPU that submits the draws).
    STRONG scaling: the work is fixed as N grows. Parity: the assembled lists on rank 0 against the unsharded oracle."""
    import torch
    import torch.distributed as dist
    from orbit_b200 import multi_gpu, scenes
    scene, view = scenes.config_c3(1.0)
    depth = scenes.make_depth(scene, view) if rank == 0 else np.zeros((view.height, view.width), np.float32)
    sv = multi_gpu.ShardedView(ctx, scene, view, depth, rank, world)
    for _ in range(2):
        sv.step(exchange=False)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t_compute = event_us(lambda: sv.step(exchange=False))
    variant = "none (one GPU: the lists are already where they are consumed)"
    if world > 1:
        sv.enable_mask_exchange(scene.n_records_lod0, scene.n_meshlet_instances)
        variant = sv.best_exchange_name()
        sv.step_best()
        torch.cuda.synchronize(); dist.barrier()
        t_full = event_us(lambda: sv.step_best())
        sv.clear_gathered()
        dist.barrier()
        sv.step_best()
        torch.cuda.synchronize(); dist.barrier()
    else:
        t_full = t_compute
        sv.step(exchange=False)
        torch.cuda.synchronize()
    t_c, t_f = max_over_ranks([t_compute[0], t_full[0]], ctx.device, world)
    out = None
    if rank == 0:
        if world > 1:
            early, late = sv.gathered_lists()
        else:
            early, late = sv.prepared.early_draws, sv.prepared.late_draws
        n_e = int(early[:4].view(torch.int32).item()); n_l = int(late[:4].view(torch.int32).item())
        ok = None
        if O is not None:
            hs = O.HostScene(scene)
            n_frames = 2 + 5 + (0 if world == 1 else 1 + 5 + 1) + 1     # every step above was one frame on the same visibility bits
            for _ in range(min(n_frames, 3)):                            # the steady state is reached after frame 1 (static camera)
                o = O.depth_prepass_culling(hs, view, depth)
            on, od = O.parse_draws(o["early"][1]); ln, ld = O.parse_draws(o["late"][1])
            ge = early[4:4 + 28 * n_e].cpu().numpy(); gl = late[4:4 + 28 * n_l].cpu().numpy()
            ok = bool(on == n_e and ln == n_l and sha(od) == sha(ge) and sha(ld) == sha(gl))
        out = {"config": "C3: 250k entities / 50M instanced meshlets, one 3840x2160 view, two-pass, entity ranges sharded over the ranks",
               "scaling": "strong", "n_gpus": world, "us_compute": t_c, "us_with_exchange": t_f, "exchange": variant,
               "value": scene.n_meshlet_instances / t_f / 1e3, "value_compute_only": scene.n_meshlet_instances / t_c / 1e3, "unit": UNIT,
               "survivors_early": n_e, "survivors_late": n_l, "list_bytes_on_rank0": 28 * (n_e + n_l), "bit_exact_vs_oracle": ok}
    sv.close()
    return out


def c5_many_view_extra(ctx, rank, world, O, n_views=256):
    """BASELINE config C5: 256 cameras over a 20 M-meshlet scene, view v on rank v mod N, no inter-GPU traffic; pass 0
    (frustum + cone) for every view. Parity: the first view of rank 0 against the oracle."""
    import torch
    import torch.distributed as dist
    from orbit_b200 import frame, multi_gpu, scenes
    from orbit_b200.passes import OcclusionCullInfo
    scene, views = scenes.config_c5(1.0, n_views=n_views)
    mine = multi_gpu.views_for_rank(len(views), rank, world)
    ds = frame.DeviceScene.upload(ctx, scene)
    infos = [frame.cull_info_for(views[v], OcclusionCullInfo("none")) for v in mine]
    pair = frame.cull_pass(ctx, "c5view", ds, infos[0])
    torch.cuda.synchronize()
    ok = None
    if rank == 0 and O is not None:
        hs = O.HostScene(scene)
        o = O.cull_pass(hs, O.gpu_cull_info(views[mine[0]], "none"))
        ghdr, grecs = frame.read_dispatch(pair[0]); ohdr, orecs = O.parse_dispatch(o[0])
        gn, gd = frame.read_draws(pair[1]); on, od = O.parse_draws(o[1])
        ok = bool(ghdr.tolist() == ohdr.tolist() and gn == on and sha(grecs) == sha(orecs) and sha(gd) == sha(od))

    def all_views():
        for info in infos:
            frame.cull_pass(ctx, "c5view", ds, info)
    all_views(); torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t = event_us(all_views, reps=3)[0]
    (t,) = max_over_ranks([t], ctx.device, world)
    if rank != 0:
        return None
    return {"config": "C5: 100k entities / 20M meshlets, %d cameras 1920x1080, pass 0 (frustum + cone), view v on rank v mod N" % len(views),
            "scaling": "strong", "n_gpus": world, "views": len(views), "us_all_views_max_rank": t, "us_per_view": t / max(len(mine), 1),
            "value": len(views) * scene.n_meshlet_instances / t / 1e3, "unit": UNIT, "bit_exact_vs_oracle_view0": ok}


# ------------------------------------------------------------------------------------------------------------
def run_ours(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    from orbit_b200 import frame, scenes
    from orbit_b200.passes import Context
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: orbit_b200 has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    ctx = Context(local_rank)
    dev = ctx.device

    scene, _ = scenes.config_c2()
    view = c2_view(scenes, scene, 0)   # every rank culls its own instance of the named C2 view (equal work per GPU: weak scaling)
    depth_np = scenes.make_depth(scene, view)

    # ---- N_COPIES independent copies of every input + view state (rotation keeps inputs out of L2)
    copies = []
    for i in range(N_COPIES):
        ds = frame.DeviceScene.upload(ctx, scene)
        vs = frame.ViewState(ctx, ds, (view.width, view.height), name="view%d" % i)
        d = torch.from_numpy(depth_np).to(dev)
        pf = frame.PreparedFrame(ctx, ds, vs, view, d, name="c%d_forward_depth_prepass" % i, main_pass=True)
        copies.append(pf)
    for pf in copies:          # frame 0 + frame 1: reach the steady state, grow scratch, then capture the graph
        pf.launch(); pf.launch()
    torch.cuda.synchronize()
    for pf in copies:
        pf.capture()
    torch.cuda.synchronize()
    code, st = ctx.poll_status()
    assert code == 0, "capacity overflow in bench"

    # ---- workload facts for the roofline (read once, outside the timed region)
    pf0 = copies[0]
    _, late_recs = frame.read_dispatch(pf0.late_dispatch)
    n_late_draws, _ = frame.read_draws(pf0.late_draws, capacity=0)
    _, early_recs = frame.read_dispatch(pf0.early_dispatch)
    n_early_draws, _ = frame.read_draws(pf0.early_draws, capacity=0)
    late_bytes, late_lanes, late_R, late_E = late_meshlet_algorithmic_bytes(late_recs, n_late_draws)
    early_lanes = int(early_recs["meshlet_count"].sum())

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- warm-up
    for i in range(max(args.warmup, 3)):
        copies[i % N_COPIES].replay()
    barrier()

    # ---- timed region: exactly K steps, CUDA events on the launching stream
    sampler = ClockSampler(local_rank)
    sampler.start()
    time.sleep(0.3)
    launches0 = ctx.launch_count
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for i in range(args.steps):
        copies[i % N_COPIES].replay()
    e1.record()
    barrier()
    step_ms = e0.elapsed_time(e1) / args.steps
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:
        last = copies[(args.steps - 1) % N_COPIES]
        passes = {k: frame.read_dispatch(getattr(last, k + "_dispatch")) + (frame.read_draws(getattr(last, k + "_draws"))[1],)
                  for k in ("early", "late", "main")}
        vs = last.vstate
        dump_outputs(args.dump_outputs, step_outputs(passes, vs.entity_visibility.cpu().numpy(), vs.meshlet_visibility.cpu().numpy(),
                                                     vs.depth_pyramid.texels.cpu().numpy()))
    if args.step_only:   # for `ncu` launch lists: the last KERNELS_PER_STEP x steps kernels of the process are exactly the timed region
        if rank == 0:
            print(json.dumps({"step_only": True, "ms_per_step": step_ms, "steps": args.steps}), flush=True)
        ctx.close()
        return
    gpu_launches = KERNELS_PER_STEP * args.steps  # (graph replays bypass the ABI counter)

    # ---- the same step again, 5 repeats of >= 50 steps each (BASELINE.md protocol: median and min), whatever --steps was
    rep_steps = max(args.steps, 50)
    rep_ms = []
    for _ in range(5):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        a.record()
        for i in range(rep_steps):
            copies[i % N_COPIES].replay()
        b.record()
        barrier()
        rep_ms.append(a.elapsed_time(b) / rep_steps)

    # ---- per-stage device times: a CUDA graph of 8 back-to-back launches of ONE stage rotating over the scene copies
    #      (no CPU in the loop, inputs out of L2), replayed several times; us per launch. The meshlet stage is two
    #      kernels (test + emit); "meshlet_*_test" times the test kernel alone (the one the roofline is quoted on).
    def time_stage(fn, reps=7, per_graph=8):
        for pf in copies:
            pf.launch()
            fn(pf, pf._stream())      # the stage itself once outside the capture: transient buffers are created (and zero-filled) here
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            for i in range(per_graph):
                pf = copies[i % N_COPIES]
                fn(pf, pf._stream())
        ts = []
        for _ in range(reps):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(); g.replay(); b.record()
            torch.cuda.synchronize()
            ts.append(a.elapsed_time(b) * 1e3 / per_graph)
        return float(np.median(ts[1:])), float(np.min(ts[1:]))

    assert all(pf.fused for pf in copies), "the C2 LATE / MAIN pair must be a compatible pair"
    stages = {"entity_early": lambda pf, s: pf.entity(False, s), "meshlet_early": lambda pf, s: pf.meshlet(False, s),
              "hiz": lambda pf, s: pf.hiz(s), "entity_late_main": lambda pf, s: pf.entity_late_main(s),
              "meshlet_late_main": lambda pf, s: pf.meshlet_late_main(s),
              # the unfused stages, for comparison (not part of the timed step)
              "unfused_entity_late": lambda pf, s: pf.entity(True, s), "unfused_meshlet_late": lambda pf, s: pf.meshlet(True, s),
              "unfused_entity_main": lambda pf, s: pf.entity("main", s), "unfused_meshlet_main": lambda pf, s: pf.meshlet("main", s)}
    k_times = {k: time_stage(fn) for k, fn in stages.items()}
    # the late-pass TEST kernel alone (the dominant kernel the roofline object is quoted on): a second context whose
    # meshlet stage skips the emit launch (ORBIT_DEBUG_SKIP=1, read at context creation; timing only — in the steady
    # state the late pass has no survivors, so skipping the emit kernel changes no buffer the next launch reads)
    os.environ["ORBIT_DEBUG_SKIP"] = "1"
    ctx_test_only = Context(local_rank)
    del os.environ["ORBIT_DEBUG_SKIP"]
    for pf in copies:
        pf.meshlet_late_main(context=ctx_test_only)     # grow that context's scratch outside the capture
    torch.cuda.synchronize()
    k_times["meshlet_late_test_kernel"] = time_stage(lambda pf, s: pf.meshlet_late_main(s, context=ctx_test_only))
    # the same kernel without the MAIN pass's bookkeeping (the LATE pass alone: what round 1's roofline was quoted on)
    k_times["meshlet_late_only_test_kernel"] = time_stage(lambda pf, s: pf.meshlet(True, s, context=ctx_test_only))
    for pf in copies:
        pf.launch()                                     # leave every copy in its steady state again
    torch.cuda.synchronize()
    # pass 0 (frustum + cone only, no Hi-Z math) over every meshlet the frustum keeps: the HBM-heaviest use of the stage
    # (extra information; the roofline object below stays on the dominant kernel of the timed step)
    from orbit_b200.passes import OcclusionCullInfo, create_meshlet_dispatch_command, create_meshlet_draw_commands
    p0 = []
    for i, pf in enumerate(copies):
        ci0 = frame.cull_info_for(pf.view, OcclusionCullInfo("none"))
        _, disp0 = create_meshlet_dispatch_command(ctx, "p0_%d" % i, pf.dscene.assets, pf.dscene.scene, ci0)
        p0.append((ci0, disp0))
    def pass0_stage(pf, s):
        i = copies.index(pf)
        create_meshlet_draw_commands(ctx, "p0_%d" % i, pf.dscene.assets, pf.dscene.scene, p0[i][0], p0[i][1])
    t_pass0 = time_stage(pass0_stage)
    _, recs0 = frame.read_dispatch(ctx._transients["p0_0_meshlet_dispatch_buffer"])
    n0, _ = frame.read_draws(ctx._transients["p0_0_meshlet_draw_command_buffer"], capacity=0)
    lanes0 = int(recs0["meshlet_count"].sum())
    bytes0 = 32 * lanes0 + 16 * len(recs0) + 12 + 64 * len(np.unique(recs0["entity_index"])) + 400 + 80 * 16 + 4 + 28 * n0

    # ---- extra: independent views in flight. The timed step above is ONE view's frame, a chain of 7 dependent,
    #      latency-bound launches; views of the same scene that do not depend on each other (shadow cascades, the
    #      256 cameras of config C5) can overlap. Same work per step as above, one context + stream + graph per scene
    #      copy, N_COPIES views in flight. Reported beside `value`, never instead of it.
    cv_ctx = [Context(local_rank) for _ in range(N_COPIES)]
    cv_streams = [torch.cuda.Stream() for _ in range(N_COPIES)]
    cv = []
    for k in range(N_COPIES):
        with torch.cuda.stream(cv_streams[k]):
            pf = frame.PreparedFrame(cv_ctx[k], copies[k].dscene, copies[k].vstate, view, copies[k].depth, name="cv%d" % k)
            pf.launch(); pf.launch()
        torch.cuda.synchronize()
        pf.capture()
        cv.append(pf)
    cv_rounds = max(args.steps // N_COPIES, 8)

    def cv_run(rounds):
        main = torch.cuda.current_stream()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(main)
        for st in cv_streams:
            st.wait_event(a)
        for _ in range(rounds):
            for k in range(N_COPIES):
                with torch.cuda.stream(cv_streams[k]):
                    cv[k].replay()
        for st in cv_streams:
            ev = torch.cuda.Event(); ev.record(st); main.wait_event(ev)
        b.record(main)
        torch.cuda.synchronize()
        return a.elapsed_time(b) / (rounds * N_COPIES)
    cv_run(4)
    barrier()
    cv_ms = min(cv_run(cv_rounds) for _ in range(3))

    # ---- end-to-end through the public API (PreparedFrame = packed C-ABI calls) with HOST buffers, software-pipelined
    #      over three streams: step i+1's pinned-host -> device input copies and compute are enqueued before the host
    #      waits for step i's survivor counts, so H2D(i+1) overlaps compute(i) and D2H(i) overlaps compute(i+1).
    #      Every step still copies its inputs in, runs the five stage calls, and reads both draw lists back.
    pin = lambda a: torch.from_numpy(np.ascontiguousarray(a).view(np.uint8).reshape(-1)).pin_memory()
    # Per-step host inputs: every entity's Transform (48 B; scene.rs:404-492 turns them into the entity buffers — here on
    # the GPU, orbit_scene_update writing straight into the buffers the culling passes read) and the depth buffer.
    from orbit_b200.scene import SceneData
    # (inputs live in write-combined pinned memory: the CPU only writes them, the copy engines read them without cache snooping)
    from orbit_b200._lib import PinnedBuffer
    wc = os.environ.get("ORBIT_BENCH_WC", "1") != "0"
    h_transforms = PinnedBuffer(scene.transforms.nbytes, write_combined=wc)
    h_transforms.array[:] = np.ascontiguousarray(scene.transforms).view(np.uint8).reshape(-1)
    h_depth = PinnedBuffer(depth_np.nbytes, write_combined=wc)
    h_depth.array[:] = depth_np.view(np.uint8).reshape(-1)
    sds = []
    for pf in copies:
        sd = SceneData(ctx, scene.n_entities)
        sd.set_entities(scene.transforms, scene.draws["mesh_index"])
        sd.entity_data_buffer, sd.entity_draw_buffer = pf.dscene.scene.entity_buffer, pf.dscene.scene.entity_draw_buffer
        sd.update_scene(pf.dscene.assets)     # first update hands out the visibility ranges (same ones as the generator's)
        sds.append(sd)
    torch.cuda.synchronize()
    assert np.array_equal(copies[0].dscene.scene.entity_draw_buffer.cpu().numpy(), scene.entity_draws), "scene update draws"
    h_count = torch.zeros(3, dtype=torch.int32).pin_memory()
    h_out_early = torch.empty(28 * scene.n_meshlet_instances, dtype=torch.uint8).pin_memory()
    h_out_late = torch.empty(28 * scene.n_meshlet_instances, dtype=torch.uint8).pin_memory()
    h_out_main = torch.empty(28 * scene.n_meshlet_instances, dtype=torch.uint8).pin_memory()
    h2d_bytes = h_transforms.numel() + h_depth.numel()
    # The loop itself is the compiled host driver (orbit_b200/host/frame_driver.cpp, the stand-in for the reference's
    # Rust host): three streams (copy-in / compute / copy-out), two steps enqueued ahead of the one being read back,
    # every GPU operation a C-ABI stage call or a cudaMemcpyAsync. A Python loop issuing the same calls spends ~185 us
    # of interpreter time per step (measured), which is as long as the step's PCIe transfers.
    e2e_steps = max(8, min(args.steps, 100))

    def e2e_run(steps, depth_resident=False):
        return frame.host_frame_loop(ctx, copies, sds, h_transforms, h_depth, h_count, h_out_early, h_out_late, h_out_main, steps,
                                     depth_resident=depth_resident)
    e2e_run(6)      # warm-up
    barrier()
    rep = e2e_run(e2e_steps)
    e2e_ms = rep["ms_per_step"]
    assert rep["h2d_bytes_per_step"] == h2d_bytes
    d2h_bytes_box = [rep["d2h_bytes_per_step"]]
    # (the entity matrices are now the ones orbit_scene_update computes in binary32, a few ulps from the generator's
    #  float64-rounded ones, so the survivor count may move by a handful of meshlets)
    assert abs(int(h_count[0]) - n_early_draws) <= max(16, n_early_draws // 100), "e2e early survivors differ from the device-resident run"
    # the same loop with the depth buffer already on the device (what Vulkan interop gives: the depth attachment is imported,
    # not copied) — reported beside `e2e`, never instead of it
    for pf in copies:
        pf.depth.copy_(torch.from_numpy(depth_np))
    e2e_run(6, depth_resident=True)
    barrier()
    rep_res = e2e_run(e2e_steps, depth_resident=True)
    e2e_res_ms = rep_res["ms_per_step"]

    # ---- extras: moving camera (C2), then the two BASELINE configs whose work is split over the ranks
    O = None
    if not args.no_parity:
        import oracle_ref as O
        O.build()
        O.lib().oracle_set_threads(os.cpu_count() or 1)      # torchrun exports OMP_NUM_THREADS=1
    moving = moving_camera_extra(ctx, frame, scenes, scene, copies, O if rank == 0 else None)

    # ---- max over ranks
    step_ms, e2e_ms, cv_ms, e2e_res_ms = max_over_ranks([step_ms, e2e_ms, cv_ms, e2e_res_ms], dev, world)
    rep_ms = max_over_ranks(rep_ms, dev, world)
    mv = max_over_ranks([moving["ms_per_step_median"], moving["ms_per_step_min"]], dev, world)
    moving["ms_per_step_median"], moving["ms_per_step_min"] = mv
    moving["value"] = scene.n_meshlet_instances * world / (mv[0] * 1e-3) / 1e9
    units = scene.n_meshlet_instances * world
    value = units / (step_ms * 1e-3) / 1e9
    e2e_value = units / (e2e_ms * 1e-3) / 1e9

    for c in cv_ctx:
        c.close()
    ctx_test_only.close()
    c3 = c5 = None
    if not args.no_configs:
        c3 = c3_sharded_extra(ctx, rank, world, O if rank == 0 else None)
        c5 = c5_many_view_extra(ctx, rank, world, O if rank == 0 else None)

    if rank == 0:
        peak, peak_src = measured_peak_gbs()
        late_us = k_times["meshlet_late_test_kernel"][0]   # the dominant kernel alone, as ncu's traffic figure is
        stage_us = k_times["meshlet_late_main"][0]         # test + emit (LATE list: empty in the steady state) + emit (MAIN list)
        achieved = late_bytes / (late_us * 1e-6) / 1e9
        cpu_baseline = None
        if world == 1 and not args.no_cpu_baseline:
            cpu_baseline = cpu_baseline_sample(scene, view, depth_np)
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": step_ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic",
            "config": {"workload": WORKLOAD,
                       "l2": "rotating %d independent copies of scene + view state (~%d MB each) so inputs come from HBM" % (
                           N_COPIES, sum(scene.bytes_summary().values()) // 2 ** 20),
                       "launch": "one CUDA graph replay per step (%d kernels: early = entity_cull + meshlet test + meshlet_emit; hiz_build; late + main fused = entity_cull + meshlet test + one meshlet_emit launch for both lists)" % KERNELS_PER_STEP,
                       "views": "every rank culls its own instance of the C2 view on a replicated scene; no data-path collective"},
            "repeats": {"what": "the timed step again, 5 repeats of %d steps each (BASELINE.md protocol)" % rep_steps,
                        "ms_per_step_median": float(np.median(rep_ms)), "ms_per_step_min": float(np.min(rep_ms)), "ms_per_step_all": rep_ms},
            "roofline": {"bound": "hbm", "kernel": "meshlet_test_direct_kernel<4,pass2,persp> (late pass, occlusion_pass=2, also filling the MAIN pass's record entries)", "achieved": achieved,
                         "peak": peak, "peak_source": peak_src, "unit": "GB/s", "frac": achieved / peak, "traffic": ncu_traffic_bytes(),
                         "traffic_source": "profiles/r2_meshlet_test_ncu.json (ncu --set full, per launch, bytes)",
                         "algorithmic_bytes_per_launch": late_bytes, "launch_us_median": late_us, "launch_us_min": k_times["meshlet_late_test_kernel"][1],
                         "stage_us_median": stage_us, "frac_stage": late_bytes / (stage_us * 1e-6) / 1e9 / peak,
                         "late_pass_alone": {"what": "the same test kernel launched for the LATE pass only (no MAIN entries / counters): the form round 1 quoted",
                                             "launch_us_median": k_times["meshlet_late_only_test_kernel"][0],
                                             "frac": late_bytes / (k_times["meshlet_late_only_test_kernel"][0] * 1e-6) / 1e9 / peak},
                         "stage": "test kernel + meshlet_emit_kernel (LATE list: nothing to emit in the steady state) + meshlet_emit_kernel (MAIN list)",
                         "lanes": late_lanes, "records": late_R, "entities": late_E, "survivors": n_late_draws,
                         "stage_gmeshlets_per_s": late_lanes / (stage_us * 1e-6) / 1e9,
                         "frac_of_nominal_8TBs": achieved / 8000.0},
            "kernels_us_median": {k: v[0] for k, v in k_times.items()},
            "hiz_build_us": k_times["hiz"][0],
            "pass0_full_sweep": {"what": "meshlet stage in pass 0 (frustum + cone, no Hi-Z) over all lanes the frustum keeps, test + emit kernels",
                                 "lanes": lanes0, "survivors": n0, "us": t_pass0[0], "algorithmic_bytes": bytes0,
                                 "achieved_GBs": bytes0 / (t_pass0[0] * 1e-6) / 1e9,
                                 "frac_of_measured_hbm": bytes0 / (t_pass0[0] * 1e-6) / 1e9 / measured_peak_gbs()[0],
                                 "stage_gmeshlets_per_s": lanes0 / (t_pass0[0] * 1e-6) / 1e9},
            "early_pass": {"lanes": early_lanes, "survivors": n_early_draws,
                           "stage_gmeshlets_per_s": early_lanes / (k_times["meshlet_early"][0] * 1e-6) / 1e9},
            "concurrent_views": {"what": "%d independent views of the scene in flight (one context + stream + CUDA graph each), depth-prepass culling only (early + Hi-Z + late)" % N_COPIES,
                                 "views_in_flight": N_COPIES, "ms_per_view": cv_ms, "value": units / (cv_ms * 1e-3) / 1e9, "unit": UNIT},
            "moving_camera": moving,
            "c3_sharded": c3, "c5_many_view": c5,
            "cpu_baseline": cpu_baseline,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(h2d_bytes), "d2h_bytes_per_step": int(d2h_bytes_box[0]),
                    "ms_per_step": e2e_ms, "steps": e2e_steps,
                    "what": "per step: pinned host entity Transforms (48 B each) + depth -> device, orbit_scene_update + 5 stage calls (C ABI: early entity + meshlet, Hi-Z, fused late + main entity / meshlet), three draw lists + counts -> host; issued by the compiled host driver (orbit_b200/host/frame_driver.cpp), software-pipelined over 3 streams (copy-in / compute / copy-out), two steps enqueued ahead of the one being read back",
                    "depth_resident": {"what": "same loop with the depth buffer already on the device (Vulkan interop imports the depth attachment instead of copying it)",
                                       "value": units / (e2e_res_ms * 1e-3) / 1e9, "ms_per_step": e2e_res_ms,
                                       "h2d_bytes_per_step": int(rep_res["h2d_bytes_per_step"]), "d2h_bytes_per_step": int(rep_res["d2h_bytes_per_step"])}},
            "gpu_launches": gpu_launches, "clocks": clocks,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    ctx.close()


def cpu_baseline_sample(scene, view, depth_np, frames=4):
    """The oracle port timed on this box's host cores: a bounded sample of the same workload (all cores: 4 frames; one
    core: 1 frame; SURVEY §8d asks for both)."""
    import oracle_ref as O
    O.build()
    O.lib().oracle_set_threads(os.cpu_count() or 1)
    hs = O.HostScene(scene)

    def frame_once():
        O.depth_prepass_culling(hs, view, depth_np)
        O.main_pass_culling(hs, view)
    for _ in range(2):
        frame_once()
    t0 = time.perf_counter()
    for _ in range(frames):
        frame_once()
    dt = (time.perf_counter() - t0) / frames
    cores = int(O.lib().oracle_threads())
    prev = O.lib().oracle_set_threads(1)
    t0 = time.perf_counter()
    frame_once()
    dt1 = time.perf_counter() - t0
    O.lib().oracle_set_threads(prev)
    return {"value": scene.n_meshlet_instances / dt / 1e9, "unit": UNIT, "cores": cores, "kind": "port",
            "ms_per_step": dt * 1e3,
            "sample": "%d whole C2 steady-state frames (early + Hi-Z + late + main) on the oracle port, OpenMP over %d host threads" % (frames, cores),
            "single_thread": {"value": scene.n_meshlet_instances / dt1 / 1e9, "ms_per_step": dt1 * 1e3, "sample": "1 frame, 1 thread"}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--step-only", action="store_true", help="stop after the timed region (profiling aid)")
    ap.add_argument("--no-configs", action="store_true", help="skip the nested C3 / C5 measurements")
    ap.add_argument("--no-parity", action="store_true", help="skip the oracle parity bits of the extras")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs as DIR/<name>.npy")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
