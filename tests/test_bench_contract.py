"""bench.py contract (CPU side): the reference arm runs without a GPU and prints ONE JSON line with the keys the
driver reads; under torchrun only rank 0 prints."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(extra_env=None):
    env = dict(os.environ)
    env.update(extra_env or {})
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1",
                        "--batch", "2"], capture_output=True, text=True, env=env, cwd=ROOT, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    return [ln for ln in r.stdout.splitlines() if ln.strip()]


def test_reference_arm_prints_one_json_line():
    lines = _run()
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "volumes/s" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["n_gpus"] == 1 and d["vs_baseline"] is None
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and "sample" in d["cpu_baseline"]
    assert d["e2e"]["value"] == d["value"] and d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert "workload" in d["config"] and "model" not in d["config"]


def test_reference_arm_other_ranks_are_silent():
    assert _run({"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"}) == []


def test_reference_arm_is_like_for_like_with_the_gpu_arm():
    """VERDICT r1 item 7: same config keys / batch as the GPU arm, the driver's --steps and --warmup honoured."""
    sys.path.insert(0, ROOT)
    import bench
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "3", "--warmup", "2",
                        "--batch", "2", "--gpus", "4"], capture_output=True, text=True, cwd=ROOT, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads(r.stdout.strip().splitlines()[-1])
    assert d["steps"] == 3 and d["warmup"] == 2 and d["n_gpus"] == 4
    assert d["config"] == bench.workload_config(bench.WORKLOADS["conf5_infer"], 2, 4, 1)
    assert set(d["config"]) == {"workload", "batch_per_gpu", "global_batch", "vis", "l2", "parallelism"}


def test_steps_below_one_are_rejected():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "0", "--batch", "2"],
                       capture_output=True, text=True, cwd=ROOT, timeout=600)
    assert r.returncode == 2 and "--steps must be at least 1" in r.stderr and r.stdout == ""


def test_dump_outputs_sample_is_fixed_and_capped(tmp_path):
    """Large outputs are written as the same seeded sample every time, 64 MB in all; small ones whole."""
    import numpy as np
    import torch
    sys.path.insert(0, ROOT)
    import bench
    arrays = {"logits": torch.randn(64, 1), "attn": torch.rand(64, 8, 65, 65), "encoded": torch.randn(1024, 65, 256)}
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), arrays)
    got = {n: np.load(tmp_path / "a" / (n + ".npy")) for n in arrays}
    assert sum(a.nbytes for a in got.values()) <= bench.DUMP_BYTES
    assert all(a.dtype == np.float32 for a in got.values())
    np.testing.assert_array_equal(got["logits"], arrays["logits"].numpy())
    np.testing.assert_array_equal(got["attn"], arrays["attn"].numpy())
    enc = arrays["encoded"].numpy().reshape(-1)
    assert 0 < got["encoded"].size < enc.size and np.isin(got["encoded"], enc).all()
    for n in arrays:
        np.testing.assert_array_equal(got[n], np.load(tmp_path / "b" / (n + ".npy")))


@pytest.mark.gpu
def test_dump_outputs_are_the_model_outputs_and_reproducible(tmp_path):
    """--dump-outputs writes the last timed step's (logits, attention weights, encoded); two runs with the same
    arguments write the same arrays, and the logits are the oracle's within the BF16 logit tolerance."""
    import numpy as np
    sys.path.insert(0, ROOT)
    from oracle import vit3d_oracle as O
    import vit3d_b200
    outs = []
    for d in ("a", "b"):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "3", "--batch", "8",
                            "--legs", "none", "--no-cpu-baseline", "--dump-outputs", str(tmp_path / d)],
                           capture_output=True, text=True, cwd=ROOT, timeout=900)
        assert r.returncode == 0, r.stderr[-2000:]
        assert json.loads(r.stdout.strip().splitlines()[-1])["steps"] == 2
        outs.append({f[:-4]: np.load(tmp_path / d / f) for f in os.listdir(tmp_path / d)})
    cfg = vit3d_b200.north_star_config(5)
    assert set(outs[0]) == {"logits", "encoded"} | {f"attn_weights_{i}" for i in range(cfg.transformer["num_layers"])}
    assert outs[0]["logits"].shape == (8, 1) and outs[0]["encoded"].shape == (8, 65, 256)
    for n, a in outs[0].items():
        np.testing.assert_allclose(outs[1][n], a, rtol=0, atol=1e-6, err_msg=n)
    lo = O.vit_forward(O.init_state_dict(cfg, seed=42), cfg, O.synth_volumes(8, seed=42))[0]
    np.testing.assert_allclose(outs[0]["logits"], lo.numpy(), rtol=0, atol=2e-2)


def test_timed_regions_do_not_call_the_oracle():
    """bench.py may use oracle/ for synthetic inputs, seeded weights and the CPU arm only - never inside a step."""
    src = open(os.path.join(ROOT, "bench.py")).read()
    body = src[src.index("def run_leg"):src.index("def ensemble_small_batch_probe")]
    step_fns = body[body.index("def pos_weight"):body.index("ms_dev, launches")]
    assert "O." not in step_fns and "oracle" not in step_fns
