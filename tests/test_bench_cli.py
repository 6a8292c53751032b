"""bench.py contract checks that need no GPU: the `--impl reference` arm prints one JSON line with
the contract's keys (it times the CPU oracle, so it runs anywhere), and the product arm fails
loudly on a machine without CUDA instead of falling back to anything."""
import json
import subprocess
import sys
from pathlib import Path

import pytest
import torch

ROOT = Path(__file__).resolve().parent.parent


def test_reference_arm_prints_the_contract_line():
    out = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                          "--workload", "tiny"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-500:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "self_training_hot_path_throughput"
    assert d["unit"] == "pixels/s" and d["higher_is_better"] is True and d["scaling"] == "weak"
    assert d["value"] > 0 and d["steps"] == 1 and d["vs_baseline"] is None and d["data"] == "synthetic"
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["cpu_baseline"]["value"] == d["value"] == d["e2e"]["value"]
    assert d["e2e"]["h2d_bytes_per_step"] == 0 == d["e2e"]["d2h_bytes_per_step"]
    assert d["config"]["workload"].startswith("tiny")


def test_reference_arm_under_torchrun_env_only_rank0_prints():
    env = dict(**__import__("os").environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1",
                          "--warmup", "0", "--workload", "tiny"], capture_output=True, text=True, timeout=600, cwd=ROOT,
                         env=env)
    assert out.returncode == 0 and not [l for l in out.stdout.splitlines() if l.startswith("{")]


@pytest.mark.skipif(torch.cuda.is_available(), reason="only meaningful on a host without CUDA")
def test_product_arm_fails_loudly_without_a_gpu():
    out = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--steps", "1", "--warmup", "0", "--workload", "tiny"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode != 0
    assert not [l for l in out.stdout.splitlines() if l.startswith("{")]


def test_both_arms_describe_the_workload_with_the_same_config_dict():
    """The driver compares the `config` of the product arm with the reference arm's."""
    sys.path.insert(0, str(ROOT))
    import bench
    from pfst_b200.synthetic import EVAL_WORKLOADS, WORKLOADS
    for name in ("cfg1", "cfg2", "cfg3", "cfg4"):
        c = bench.config_dict(WORKLOADS[name])
        assert c["workload"] == WORKLOADS[name].name and c["params"] > 43_000_000
    assert bench.config_dict(WORKLOADS["cfg2"])["params"] == 43579868
    assert bench.eval_config_dict(EVAL_WORKLOADS["cfg5"])["maps"] == 10000


def test_dump_outputs_writes_float_arrays_and_samples_large_ones_alike(tmp_path):
    """--dump-outputs: every array lands as float32/float64 .npy; a large one is replaced by the same
    seeded sample on every call, so two runs of two builds can be compared element for element."""
    sys.path.insert(0, str(ROOT))
    import numpy as np
    import bench
    big = torch.arange(bench.DUMP_MAX_ELEMS + 12345, dtype=torch.int64)
    arrays = {"loss": torch.tensor([1.5, 2.5]), "label": torch.tensor([[0, 3], [255, 7]], dtype=torch.uint8),
              "big": big}
    for d in (tmp_path / "a", tmp_path / "b"):
        bench.dump_outputs(d, arrays)
    a = {p.stem: np.load(p) for p in (tmp_path / "a").glob("*.npy")}
    assert sorted(a) == ["big", "label", "loss"]
    assert a["loss"].dtype == np.float32 and a["label"].dtype == np.float32 and a["big"].dtype == np.float64
    assert np.array_equal(a["label"], [[0, 3], [255, 7]])
    assert a["big"].shape == (bench.DUMP_MAX_ELEMS,) and np.all(np.diff(a["big"]) >= 0)
    assert np.array_equal(a["big"], np.load(tmp_path / "b" / "big.npy"))


def test_steps_below_one_and_dumps_of_the_reference_arm_are_rejected():
    for extra in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "unused"]):
        out = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--workload", "tiny", *extra],
                             capture_output=True, text=True, timeout=600, cwd=ROOT)
        assert out.returncode == 2 and "error" in out.stderr, extra


def test_eval_sweep_reference_arm():
    out = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                          "--workload", "tiny_eval"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-500:]
    d = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][0])
    assert d["metric"] == "miou_eval_sweep_throughput" and d["scaling"] == "strong" and d["dtype"] == "int64"
    assert d["value"] > 0 and d["config"]["maps"] == 8
