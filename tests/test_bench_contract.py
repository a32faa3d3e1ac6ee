"""bench.py's reference arm on the CPU (the part of the bench contract that runs without a GPU): one JSON line with
`impl: reference`, exactly K timed steps after the same warm-up count our own arm reports, the metric / unit / config
of our arm, and the `cpu_baseline` / `e2e` objects the driver reads."""
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_the_contract_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "1"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["steps"] == 2 and line["warmup"] == 3      # W >= 3, like our arm
    assert line["unit"] == "tokens/s" and line["higher_is_better"] is True and line["value"] > 0
    assert line["config"]["seq_len"] == 4096 and line["config"]["heads"] == 32 and line["config"]["global_batch"] == 8
    assert line["cpu_baseline"]["kind"] in ("port", "reference") and line["cpu_baseline"]["value"] == line["value"]
    assert line["e2e"] == {"value": line["value"], "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    # a step is a bounded sample, timed as it is: ms_per_step x tokens/s = the tokens of one sample
    assert abs(line["ms_per_step"] * 1e-3 * line["value"] - line["tokens_per_step"]) <= 1e-6 * line["tokens_per_step"]
    assert line["gpu_launches"] == 0


def test_bad_arguments_are_refused(tmp_path):
    for extra in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", str(tmp_path)]):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *extra], capture_output=True, text=True,
                             timeout=120, cwd=ROOT)
        assert out.returncode == 2 and out.stdout == "", extra
    assert os.listdir(tmp_path) == []


def test_dump_index_is_a_fixed_sample_without_repeats():
    import bench
    idx = bench.dump_index()
    assert idx.numel() == bench.DUMP_SAMPLE and (idx[1:] > idx[:-1]).all()
    assert 0 <= idx[0] and idx[-1] < bench.B * bench.T * bench.C
    assert torch.equal(idx, bench.dump_index())


def test_ranks_other_than_zero_do_no_work_in_the_reference_arm():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "2"],
                         capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""
