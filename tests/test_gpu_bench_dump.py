"""bench.py --dump-outputs: the files hold, bit for bit, what RUN_CUDA_RWKV6 + backward returns to a caller on the
benchmark's inputs, within bench.py's size bound.  Every timed step runs on the same inputs, so this cannot tell the
last step's results from an earlier one's.  `pytest -m gpu`."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_outputs_hold_the_step_results(tmp_path):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "3", "--warmup", "1",
                          "--no-e2e", "--no-bi-encoder", "--no-sft", "--no-cpu-baseline", "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-3000:]
    assert json.loads(out.stdout.strip().splitlines()[-1])["steps"] == 3
    names = ("y", "gr", "gk", "gv", "gw", "gu")
    assert sorted(os.listdir(tmp_path)) == sorted(n + ".npy" for n in names)
    assert sum(os.path.getsize(tmp_path / (n + ".npy")) for n in names) <= 64 << 20
    got = {n: np.load(tmp_path / (n + ".npy")) for n in names}
    assert all(a.dtype == np.float32 for a in got.values())

    import bench
    import rwkv_lm_ext_b200 as M
    from rwkv_lm_ext_b200.synthetic import make_inputs
    r, k, v, w, u, gy = make_inputs(bench.B, bench.T, bench.H, seed=0, decay="model", device="cuda")
    leaves = [t.requires_grad_(True) for t in (r, k, v, w, u)]
    y = M.RUN_CUDA_RWKV6(bench.B, bench.T, bench.C, bench.H, *leaves)
    y.backward(gy)
    idx = bench.dump_index("cuda")
    want = [y.detach()] + [t.grad for t in leaves[:4]]
    for n, t in zip(names, want):
        assert np.array_equal(got[n], t.reshape(-1)[idx].float().cpu().numpy()), n
    assert np.array_equal(got["gu"], leaves[4].grad.float().cpu().numpy())
