"""CPU: the reference arm of bench.py (`--impl reference` = the oracle port on the host cores) runs without a GPU and
prints one JSON line with every key the bench contract names. GPU: what `--dump-outputs` writes for the timed path
equals what the reference arm writes for the same step."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PASSES = ("early", "late", "main")
DUMPED = ["%s_%s" % (k, a) for k in PASSES for a in ("dispatch_header", "dispatch_records", "draw_count", "draw_commands")] + [
    "entity_visibility", "meshlet_visibility", "hiz_texels"]


def _load_dump(d):
    dumped = {f[:-4]: np.load(os.path.join(d, f)) for f in os.listdir(d) if f.endswith(".npy")}
    assert set(dumped) <= set(DUMPED) and {"entity_visibility", "meshlet_visibility", "hiz_texels"} <= set(dumped)
    assert all(a.size > 0 and a.dtype in (np.float32, np.float64) for a in dumped.values())
    assert sum(a.nbytes for a in dumped.values()) <= 64 * 2 ** 20
    for k in PASSES:        # a list is written exactly when its count says it has entries
        n_records, n_draws = int(dumped[k + "_dispatch_header"][0]), int(dumped[k + "_draw_count"][0])
        assert len(dumped.get(k + "_dispatch_records", ())) == n_records and len(dumped.get(k + "_draw_commands", ())) == n_draws, k
    return dumped


def test_reference_arm_prints_contract_line(tmp_path):
    env = dict(os.environ, OMP_NUM_THREADS="4")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "1", "--steps", "1", "--warmup", "1",
                          "--dump-outputs", str(tmp_path)], capture_output=True, text=True, env=env, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in line, k
    assert line["impl"] == "reference" and line["higher_is_better"] is True and line["vs_baseline"] is None
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0
    assert line["value"] > 0 and "workload" in line["config"]
    dumped = _load_dump(tmp_path)
    assert dumped["early_draw_count"][0] > 0 and dumped["early_dispatch_header"][0] > 0


def test_reference_arm_is_silent_on_other_ranks():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "1"],
                         capture_output=True, text=True, env=env, timeout=120)
    assert out.returncode == 0 and out.stdout.strip() == ""


@pytest.mark.gpu
def test_dumped_outputs_of_timed_path_match_reference_arm(tmp_path):
    """Every dumped array, exactly. In the C2 steady state the late pass emits nothing, so its lists are compared through
    their count and dispatch header only (late lists with entries are checked by tests/test_gpu_late_main.py)."""
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    dumps = {}
    for impl, extra in (("ours", ["--step-only"]), ("reference", [])):      # 3 steps: the last one runs on scene copy 2, not 0
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", impl, "--gpus", "1", "--steps", "3", "--warmup", "1",
                              "--dump-outputs", str(tmp_path / impl)] + extra, capture_output=True, text=True, timeout=600)
        assert out.returncode == 0, out.stderr[-2000:]
        dumps[impl] = _load_dump(tmp_path / impl)
    assert set(dumps["ours"]) == set(dumps["reference"])
    for name, a in dumps["ours"].items():
        assert a.dtype == dumps["reference"][name].dtype, name
        assert np.array_equal(a, dumps["reference"][name]), name
    assert dumps["ours"]["main_draw_count"][0] > 0
