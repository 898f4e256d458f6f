"""bench.py's reference arm (`--impl reference`: the CPU restatement of the path on the host cores) runs without a
GPU, so its JSON contract is checked here; under a multi-rank launch only rank 0 prints.  On a GPU: --dump-outputs
writes what the last timed step of the native arm computed."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench(flags, extra_env=None):
    env = dict(os.environ, **(extra_env or {}))
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *flags], capture_output=True, text=True,
                       timeout=600, env=env, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    return [ln for ln in r.stdout.splitlines() if ln.strip()]


def _run(extra_env=None, *flags):
    return _bench(["--impl", "reference", "--steps", "2", "--warmup", "1", "--cpu-sample", "2000", *flags], extra_env)


def test_reference_arm_prints_one_json_line_with_the_contract_keys():
    lines = _run()
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "flow_log_prob_events_per_s" and d["unit"] == "events/s"
    assert d["higher_is_better"] is True and d["steps"] == 2 and d["warmup"] == 1 and d["value"] > 0
    assert d["config"]["workload"] == "bounded16" and d["config"]["D"] == 16 and d["config"]["K"] == 32
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("port", "reference") and cb["cores"] >= 1 and cb["value"] == d["value"] and "sample" in cb
    assert d["e2e"] == {"value": d["value"], "unit": "events/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["vs_baseline"] is None and d["gpu_launches"] == 0


def test_reference_arm_other_ranks_exit_quietly():
    assert _run({"RANK": "1", "LOCAL_RANK": "1", "WORLD_SIZE": "2"}, "--gpus", "2") == []


@pytest.mark.gpu
def test_dump_outputs_hold_the_last_timed_step(tmp_path):
    """--dump-outputs DIR: DIR/log_prob.npy is the float32 log_prob of the last of the --steps timed steps, bit for bit
    what Flow.__call__ gives on that step's seeded inputs (steps 3 after warmup 3: input set 5, seed 1000 + 5)."""
    import torch

    import bench

    M = 5000
    lines = _bench(["--steps", "3", "--warmup", "3", "--batch", str(M), "--no-extras", "--train-batch", "0",
                    "--cpu-sample", "2000", "--dump-outputs", str(tmp_path)])
    assert len(lines) == 1 and json.loads(lines[0])["steps"] == 3
    assert sorted(os.listdir(tmp_path)) == ["log_prob.npy"]
    got = np.load(tmp_path / "log_prob.npy")
    assert got.dtype == np.float32 and got.shape == (M,)

    w = dict(bench.WORKLOADS["bounded16"], M=M)
    flow, variables = bench.build_flow(w, torch.device("cuda", 0))
    x, _ = bench.synth(w, M, 1000 + 5)
    want = flow.apply(variables, torch.from_numpy(x).cuda()).cpu().numpy()
    np.testing.assert_array_equal(got, want)
