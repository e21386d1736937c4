"""GPU parity of the tcgen05 (3xTF32) weight gradient vs the CPU oracle."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def rel_linf(a, b):
    a = np.asarray(a, dtype=np.float64); b = np.asarray(b, dtype=np.float64)
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-30))


def cu(x):
    return torch.as_tensor(np.ascontiguousarray(x, dtype=np.float32)).cuda()


WG_CASES = [
    # n, h, w, cin, cout, k, dil
    (1, 16, 32, 64, 32, 3, 1), (1, 24, 48, 128, 128, 3, 1), (2, 24, 40, 128, 96, 3, 4), (1, 16, 32, 72, 128, 3, 1),
    (1, 12, 40, 136, 128, 3, 1), (1, 32, 64, 64, 32, 3, 1), (2, 16, 20, 192, 192, 3, 1), (1, 16, 16, 128, 64, 1, 1),
    (1, 96, 320, 128, 128, 3, 1),
]


@pytest.mark.parametrize('case', WG_CASES)
def test_wgrad_tc(case):
    from madstereo import ops
    from oracle import tf1_ops as T
    n, h, w, cin, cout, k, dil = case
    rng = np.random.default_rng(sum(case))
    x = rng.standard_normal((n, h, w, cin)).astype(np.float32)
    g = rng.standard_normal((n, h, w, cout)).astype(np.float32)
    wt = torch.zeros(k, k, cin, cout, requires_grad=True)
    bt = torch.zeros(cout, requires_grad=True)
    pre = T.conv2d(torch.tensor(x), wt, bt, stride=1, dilation=dil, alpha=None)
    gw, gb = torch.autograd.grad(pre, [wt, bt], grad_outputs=torch.tensor(g))
    dw, db = ops.conv2d_wgrad_tc(cu(x), cu(g), k, k, dil)
    torch.cuda.synchronize()
    assert rel_linf(dw.cpu().numpy(), gw.numpy()) < 5e-5, 'dw'
    assert rel_linf(db.cpu().numpy(), gb.numpy()) < 5e-5, 'db'
