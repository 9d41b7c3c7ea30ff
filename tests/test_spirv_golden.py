"""CPU: the oracle against outputs of the REFERENCE'S OWN SHIPPED SHADERS (tests/golden/spirv_reference.json, produced
in the build container by running /root/reference/shaders/*.comp.spv in the SPIR-V interpreter oracle/spirv_vm — see
tests/golden/make_spirv_golden.py). This is what pins the oracle: Hi-Z pyramids and visibility words byte for byte,
dispatch records / draw commands / cluster lists as sorted sets (the shaders append with atomicAdd)."""
import json
import os

import numpy as np
import pytest

import spirv_cases as S

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def golden():
    with open(os.path.join(ROOT, "tests", "golden", "spirv_reference.json")) as f:
        return json.load(f)


def test_hiz_pyramids_match_shipped_depth_reduce(oracle, golden):
    for name, depth in S.hiz_cases().items():
        _, tex = oracle.hiz_build(depth)
        assert S.matches(golden["hiz"][name], np.asarray(tex).reshape(-1)), name


def test_cull_passes_match_shipped_entity_and_meshlet_shaders(oracle, golden):
    for name, case in S.cull_cases().items():
        g = golden["cull"][name]
        sc, view, depth, mocc, frames, protocol = case
        hs = oracle.HostScene(sc)
        k = 0
        for f in range(frames):
            passes = {"two_pass": [("early", "read"), ("late", "write")], "pass0": [("pass0", "none")], "pass2_only": [("late", "write")]}[protocol]
            for label, kind in passes:
                if kind == "write":
                    hs.update_pyramid(depth)
                out = oracle.cull_pass(hs, S.tweak_gpu_cull_info(oracle.gpu_cull_info(view, kind, mocc), name))
                step = g["steps"][k]; k += 1
                assert (step["frame"], step["pass"]) == (f, label)
                hdr, recs = S.canon_records(out[0])
                n, draws = S.canon_draws(out[1])
                assert hdr == step["dispatch_header"], (name, f, label)
                assert S.matches(step["records"], recs), (name, f, label, "records")
                assert n == step["draw_count"] and S.matches(step["draws"], draws), (name, f, label, "draws")
                assert S.matches(step["entity_visibility"], hs.entity_visibility), (name, f, label, "entity visibility")
                assert S.matches(step["meshlet_visibility"], hs.meshlet_visibility), (name, f, label, "meshlet visibility")
        if g["hiz"] is not None:
            assert S.matches(g["hiz"], hs.hiz_texels.reshape(-1)), (name, "hiz")
        assert sum(s["draw_count"] for s in g["steps"]) > 0


def test_clusters_match_shipped_light_cluster_shaders(oracle, golden):
    for name, (p, depth, lights) in S.cluster_cases().items():
        g = golden["clusters"][name]
        c = S.canon_clusters(oracle.light_cluster(p, depth, lights))
        assert c["header"] == g["header"] and c["total"] == g["total"], name
        for k in ("masks", "bounds", "active", "counts", "lists"):
            assert S.matches(g[k], c[k]), (name, k)
    assert max(S.unpack(golden["clusters"]["cap_256"]["counts"], np.uint32)) == 256     # the MAX_LIGHTS_PER_CLUSTER cap was exercised


def test_task_payloads_match_shipped_task_shaders(oracle, golden):
    """forward_depth_prepass.task / forward.task / shadow.task (shipped SPIR-V, interpreted) vs the oracle's payload output."""
    cases = S.cull_cases()
    for name, kind in (("ortho_pass0", "none"), ("ortho_pass2", "write"), ("persp_two_pass_entity_occlusion_only", "write")):
        sc, view, depth, mocc, _, _ = cases[name]
        hs = oracle.HostScene(sc)
        if kind == "write":
            hs.update_pyramid(depth)
        out = oracle.cull_pass(hs, oracle.gpu_cull_info(view, kind, mocc), task_payloads=True)
        nrec = int(out[0][:4].view(np.uint32)[0])
        pl = S.canon_payload_buffer(out[2], nrec)
        for shader, entry in golden["task"][name].items():
            assert S.matches(entry["payloads"], pl), (name, shader)
            assert int(pl["task_count"].sum()) == entry["tasks"] > 0
            if "meshlet_visibility_comp_semantics" in entry:
                assert S.matches(entry["meshlet_visibility_comp_semantics"], hs.meshlet_visibility), (name, shader, "visibility")
