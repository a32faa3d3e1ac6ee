"""One process driving two devices in turn (per-device kernel attributes and memory pools).  Needs two
GPUs: skipped on a single-GPU box.  `pytest -m gpu`."""
import pytest
import torch

from tests.util import make_inputs

pytestmark = pytest.mark.gpu


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_two_devices_in_one_process():
    import rwkv_lm_ext_b200 as M
    B, T, H = 2, 2304, 3                      # long enough for the time-segmented training pair
    C = H * 64
    outs = []
    for dev in ("cuda:0", "cuda:1", "cuda:0"):
        with torch.cuda.device(dev):
            r, k, v, w, u, gy = make_inputs(B, T, H, 3, decay="model", device=dev)
            ts = [t.clone().requires_grad_(True) for t in (r, k, v, w, u)]
            y = M.RUN_CUDA_RWKV6(B, T, C, H, *ts)
            y.backward(gy)
            layer = M.Tmix_x060(C, H).bfloat16().to(dev)
            x = torch.randn(B, 64, C, device=dev).bfloat16().requires_grad_(True)
            layer(x).float().sum().backward()
            torch.cuda.synchronize()
            outs.append([y.detach().cpu()] + [t.grad.cpu() for t in ts])
    for other in (outs[1], outs[2]):
        for a, b in zip(outs[0], other):
            assert torch.equal(a, b)
