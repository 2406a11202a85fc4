"""CPU-only: the reference arm of bench.py (`--impl reference`, the CPU restatement on the host cores) prints ONE JSON
line with the contract's keys; ranks other than 0 print nothing and exit 0; the reference's shaders run outside the tests."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(env_extra=None):
    env = dict(os.environ)
    env.update(env_extra or {})
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "1", "--steps", "1", "--warmup", "0", "--cpu-sample-draws", "3000", "--draws", "3000", "--depth", "256"]
    return subprocess.run(cmd, capture_output=True, text=True, env=env, timeout=600)


def test_reference_arm_json_contract():
    res = _run()
    assert res.returncode == 0, res.stderr[-2000:]
    lines = [l for l in res.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in d, key
    assert d["impl"] == "reference" and d["higher_is_better"] is True and d["vs_baseline"] is None and d["data"] == "synthetic"
    assert d["value"] > 0 and d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0 and d["e2e"]["value"] == d["value"]
    assert "workload" in d["config"]
    # the reference's own shaders, timed by a child process where they are built (informational)
    import refshader_lib

    shaders = d["cpu_baseline"]["reference_shaders"]
    assert (shaders["value"] > 0) if refshader_lib.available() else ("unavailable" in shaders), shaders


def test_reference_shader_path_outside_a_pinned_test():
    """bench.py drives RefShaderPath outside any test: with the reference's shaders it runs them (and agrees with the oracle);
    without them it refuses, instead of standing in for them with nothing to hold the stand-in to."""
    import numpy as np
    import pytest

    import oracle_lib
    import refshader_lib
    from niagara_b200 import scenes

    s = scenes.instanced_scene(os.path.join(ROOT, "tests", "golden", "kitten.nvcg"), 256)
    if not refshader_lib.available():
        with pytest.raises(RuntimeError):
            refshader_lib.RefShaderPath(s.meshes, s.meshlets, s.draws, *s.screen)
        return
    r = refshader_lib.RefShaderPath(s.meshes, s.meshlets, s.draws, *s.screen)
    o = oracle_lib.OraclePath(s.meshes, s.meshlets, s.draws, *s.screen)
    for p in (r, o):
        p.set_visibility_bits(s.visibility_bits)
        p.frame(s.cull_data(), s.depth, cluster_backface=True)
    assert np.array_equal(r.dccb, o.dccb) and np.array_equal(r.ccb, o.ccb) and np.array_equal(r.mvb, o.mvb)


def test_reference_arm_other_ranks_are_silent():
    res = _run({"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"})
    assert res.returncode == 0 and res.stdout.strip() == ""
