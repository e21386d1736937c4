"""GPU parity: every CUDA op (through the C ABI) vs the CPU oracle on seeded random tensors."""
import os

import numpy as np
import pytest
import torch

from conftest import ROOT

pytestmark = pytest.mark.gpu


def rel_linf(a, b):
    a = np.asarray(a, dtype=np.float64); b = np.asarray(b, dtype=np.float64)
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-30))


def cu(x):
    return torch.as_tensor(np.ascontiguousarray(x, dtype=np.float32)).cuda()


@pytest.fixture(scope='module')
def ops():
    from madstereo import ops as o
    return o


def _oracle():
    from oracle import tf1_ops as T
    return T


# shapes: MADNet levels (SURVEY §8a a1) at 1280x384 for the small ones, reduced width for the big ones
CORR_SHAPES = [(1, 6, 20, 192, 2, 1), (1, 12, 40, 128, 2, 1), (2, 24, 80, 96, 2, 1), (1, 48, 160, 64, 2, 1),
               (1, 96, 320, 32, 2, 1), (1, 8, 24, 32, 4, 2), (1, 5, 7, 8, 2, 1)]


@pytest.mark.parametrize('shape', CORR_SHAPES)
@pytest.mark.parametrize('warp', [False, True])
def test_correlation_fwd_bwd(ops, shape, warp):
    T = _oracle()
    b, h, w, c, d, s = shape
    rng = np.random.default_rng(hash(shape) % 1000)
    x = rng.standard_normal((b, h, w, c)).astype(np.float32)
    y = rng.standard_normal((b, h, w, c)).astype(np.float32)
    u = (rng.uniform(-3.0, 3.0, (b, h, w, 1))).astype(np.float32) if warp else None
    if warp:
        u[0, 0, 0, 0] = -7.25; u[0, -1, -1, 0] = 9.5          # far outside on both borders
    xt = torch.tensor(x, requires_grad=True); yt = torch.tensor(y, requires_grad=True)
    ut = torch.tensor(u, requires_grad=True) if warp else None
    yw = T.linear_warp(yt, ut) if warp else yt
    ref = T.correlation(xt, yw, d, s)
    out = ops.correlation(cu(x), cu(y), d, s, u=cu(u) if warp else None)
    assert rel_linf(out.cpu().numpy(), ref.detach().numpy()) < 2e-5
    g = rng.standard_normal(ref.shape).astype(np.float32)
    grads = torch.autograd.grad(ref, [xt, yt] + ([ut] if warp else []), grad_outputs=torch.tensor(g))
    dx, dy, du = ops.correlation_bwd(cu(x), cu(y), cu(g), d, s, u=cu(u) if warp else None, want_du=warp)
    assert rel_linf(dx.cpu().numpy(), grads[0].numpy()) < 2e-5
    assert rel_linf(dy.cpu().numpy(), grads[1].numpy()) < 2e-5
    if warp:
        assert rel_linf(du.cpu().numpy(), grads[2].numpy()) < 1e-4


@pytest.mark.parametrize('shape', [(1, 12, 40, 32, 2.0), (2, 5, 136, 64, 3.0), (1, 3, 300, 32, 70.0), (1, 4, 72, 96, 40.0)])
def test_cost_volume_concat(ops, shape):
    """Fused warp + correlation + concat (MadNet.py:370-375): multi-tile rows, a ragged last tile, and warp offsets wide
    enough that taps leave the staged right-feature window (the kernel's direct-from-global path)."""
    T = _oracle()
    b, h, w, c, umax = shape
    rng = np.random.default_rng(1)
    x = rng.standard_normal((b, h, w, c)).astype(np.float32)
    y = rng.standard_normal((b, h, w, c)).astype(np.float32)
    u = rng.uniform(-umax, umax, (b, h, w, 1)).astype(np.float32)
    ref = torch.cat([torch.tensor(x), T.correlation(torch.tensor(x), T.linear_warp(torch.tensor(y), torch.tensor(u)), 2),
                     torch.tensor(u)], -1)
    out = ops.cost_volume(cu(x), cu(y), 2, 1, u=cu(u))
    assert out.shape == ref.shape
    assert rel_linf(out.cpu().numpy(), ref.numpy()) < 2e-5
    plain = ops.correlation(cu(x), cu(y), 2, 1, u=cu(u))
    assert rel_linf(plain.cpu().numpy(), ref.numpy()[..., c:c + 5]) < 2e-5


WIDE_SHAPES = [(1, 12, 40, 128, 40), (1, 5, 100, 64, 40), (2, 7, 70, 48, 20), (1, 3, 64, 16, 8), (1, 96, 320, 128, 40)]


@pytest.mark.parametrize('shape', WIDE_SHAPES)
def test_correlation_wide_window(ops, shape):
    """DispNet's 81-displacement correlation on the banded tensor-core kernel (csrc/corr_mma.cu) vs the oracle; also through
    the generic entry point (same numbers as the CUDA-core kernel within the same tolerance)."""
    T = _oracle()
    b, h, w, c, d = shape
    rng = np.random.default_rng(sum(shape))
    x = (rng.standard_normal((b, h, w, c)) * 3.0).astype(np.float32)
    y = (rng.standard_normal((b, h, w, c)) * 3.0).astype(np.float32)
    ref = T.correlation(torch.tensor(x), torch.tensor(y), d, 1).numpy()
    out = ops.correlation_wide(cu(x), cu(y), d, act_scale=64.0)
    torch.cuda.synchronize()
    assert out.shape == ref.shape
    assert rel_linf(out.cpu().numpy(), ref) < 2e-5
    plain = ops.correlation(cu(x), cu(y), d, 1)
    assert rel_linf(plain.cpu().numpy(), ref) < 2e-5
    # into a wider buffer (the engine writes channels [0, 81) of a 148-channel concat buffer): neighbours untouched
    buf = torch.full((b, h, w, 2 * d + 1 + 7), 7.0, device='cuda')
    ops.correlation_wide(cu(x), cu(y), d, act_scale=64.0, out=buf)
    torch.cuda.synchronize()
    assert rel_linf(buf[..., :2 * d + 1].cpu().numpy(), ref) < 2e-5
    assert bool((buf[..., 2 * d + 1:] == 7.0).all())


@pytest.mark.parametrize('shape', [(1, 12, 40, 128, 40), (1, 5, 100, 64, 40), (2, 7, 70, 32, 20), (1, 24, 320, 128, 40)])
def test_correlation_wide_window_bwd(ops, shape):
    """Gradients of the 81-displacement correlation: two banded products on mma.sync tiles with bf16 hi/lo operands
    (csrc/corr_mma.cu) -- the arithmetic class of the convolution gradients, tolerance 1e-4 relative L-inf."""
    T = _oracle()
    b, h, w, c, d = shape
    rng = np.random.default_rng(sum(shape) + 1)
    x = rng.standard_normal((b, h, w, c)).astype(np.float32)
    y = rng.standard_normal((b, h, w, c)).astype(np.float32)
    xt = torch.tensor(x, requires_grad=True); yt = torch.tensor(y, requires_grad=True)
    ref = T.correlation(xt, yt, d, 1)
    g = (rng.standard_normal(ref.shape) * 1e-3).astype(np.float32)          # gradient-sized values: no fixed scale to rely on
    gx, gy = torch.autograd.grad(ref, [xt, yt], grad_outputs=torch.tensor(g))
    dx, dy, _ = ops.correlation_bwd(cu(x), cu(y), cu(g), d, 1)
    torch.cuda.synchronize()
    assert rel_linf(dx.cpu().numpy(), gx.numpy()) < 1e-4
    assert rel_linf(dy.cpu().numpy(), gy.numpy()) < 1e-4


# Output and kernel time of the reference's own CorrelateData kernel (compiled unmodified for sm_100a), recorded on a B200
# by tests/golden/make_reference_corr_golden.py.
REF_CORR_GOLDEN = os.path.join(ROOT, 'tests', 'golden', 'reference_corr_native.npz')


def _corr_inputs(b, h, w, c, seed):
    """The inputs of the recorded timing shapes (same generator as make_reference_corr_golden.py)."""
    g = torch.Generator().manual_seed(seed)
    return torch.randn(b, h, w, c, generator=g), torch.randn(b, h, w, c, generator=g)


def test_correlation_matches_reference_native_kernel(ops):
    """The reference's own CorrelateData kernel on padded inputs: its recorded output."""
    g = np.load(REF_CORR_GOLDEN)
    d = (g['exact_out'].shape[-1] - 1) // 2
    mine = ops.correlation(cu(g['exact_x']), cu(g['exact_y']), d)
    assert rel_linf(mine.cpu().numpy(), g['exact_out']) < 2e-5


def test_correlation_speed_vs_reference_native_kernel(ops):
    """SURVEY 8(d): the reference's own CorrelateData kernel is "the kernel to beat" on the same GPU.  Its time on a B200
    (pre-padded inputs, kernel only: its tf.pad / tf.transpose round trips are not charged) and a seeded sample of its
    output are recorded in tests/golden/reference_corr_native.npz; ours is timed here on the unpadded NHWC tensors."""
    g = np.load(REF_CORR_GOLDEN)
    shapes = {'madnet_L6_1280x384': (1, 6, 20, 192, 2), 'madnet_L5': (1, 12, 40, 128, 2), 'madnet_L4': (1, 24, 80, 96, 2),
              'madnet_L3': (1, 48, 160, 64, 2), 'madnet_L2': (1, 96, 320, 32, 2), 'madnet_L2_1920x1088_B8': (8, 272, 480, 32, 2),
              'dispnet_1280x384': (1, 96, 320, 128, 40)}
    flush = torch.empty(256 << 20, dtype=torch.uint8, device='cuda')

    def timeit(fn):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        ts = []
        for _ in range(7):
            flush.zero_()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); fn(); e1.record(); torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1) * 1e3)
        ts.sort()
        return ts[len(ts) // 2]

    rows = {}
    for name, (b, h, w, c, d) in shapes.items():
        x, y = _corr_inputs(b, h, w, c, int(g[name + '_seed']))
        assert np.array_equal(x.view(-1)[:16].numpy(), g[name + '_x_probe']), 'inputs differ from the recorded ones: ' + name
        x, y = x.cuda(), y.cuda()
        mine = torch.empty(b, h, w, 2 * d + 1, device='cuda')
        if d >= 8:      # DispNet: the banded tensor-core kernel the engine runs (fp16 hi/lo, activation scale 64)
            t_mine = timeit(lambda: ops.correlation_wide(x, y, d, 64.0, out=mine))
        else:
            t_mine = timeit(lambda: ops.correlation_into(x, y, d, mine))
        got = mine.view(-1)[torch.from_numpy(g[name + '_index']).cuda()].cpu().numpy().astype(np.float64)
        assert np.abs(got - g[name + '_sample']).max() / max(float(g[name + '_absmax']), 1e-30) < 2e-5, name
        t_ref = float(g[name + '_reference_us'])
        byts = b * h * w * (2 * c + 2 * d + 1) * 4
        rows[name] = {'reference_us': t_ref, 'ours_us': t_mine, 'speedup': t_ref / t_mine, 'bytes': byts,
                      'ours_gbs': byts / t_mine / 1e3, 'reference_gbs': byts / t_ref / 1e3}
    print('reference timed on', g['device'], rows)
    assert rows['madnet_L2_1920x1088_B8']['speedup'] > 1.0 and rows['dispnet_1280x384']['speedup'] > 1.0, rows


CONV_CASES = [
    # n, h, w, cin, cout, k, stride, dil, alpha
    (2, 32, 64, 3, 16, 3, 2, 1, 0.2), (2, 16, 32, 16, 16, 3, 1, 1, 0.2), (1, 16, 32, 16, 32, 3, 2, 1, 0.2),
    (1, 12, 40, 134, 128, 3, 1, 1, 0.2), (1, 24, 40, 128, 96, 3, 1, 1, 0.2), (1, 24, 40, 32, 1, 3, 1, 1, 1.0),
    (1, 24, 40, 33, 128, 3, 1, 1, 0.2), (1, 24, 48, 128, 128, 3, 1, 4, 0.2), (1, 24, 48, 96, 64, 3, 1, 16, 0.2),
    (1, 17, 23, 20, 24, 3, 2, 1, 0.1), (1, 32, 32, 3, 64, 7, 2, 1, 0.1), (1, 16, 16, 64, 128, 5, 2, 1, 0.1),
    (1, 16, 16, 128, 64, 1, 1, 1, 0.1), (1, 6, 20, 197, 128, 3, 1, 1, 0.2),
    # full-resolution pyramid layers (direct small-channel kernels, csrc/conv_small.cu): >= 4096 output pixels, odd widths
    (2, 96, 130, 3, 16, 3, 2, 1, 0.2), (1, 70, 72, 16, 16, 3, 1, 1, 0.2), (1, 65, 67, 3, 16, 3, 1, 1, 1.0),
    (1, 68, 64, 8, 16, 3, 1, 2, 0.2),
    # single output channel: weight gradient through the dedicated head kernel (csrc/conv_head.cu:conv_head_wgrad) --
    # 8 / 16 / 256 lanes per pixel, a channel count that is not a multiple of 4, and the 4x4 stride-2 1 -> 1 geometry of
    # DispNet's up_predict gradient
    (2, 20, 36, 64, 1, 3, 1, 1, 1.0), (1, 6, 20, 1024, 1, 3, 1, 1, 1.0), (1, 9, 11, 5, 1, 3, 1, 2, 1.0),
    (2, 16, 24, 1, 1, 4, 2, 1, 1.0), (1, 192, 640, 32, 1, 3, 1, 1, 1.0),
]


@pytest.mark.parametrize('case', CONV_CASES)
def test_conv2d_fwd_dgrad_wgrad(ops, case):
    T = _oracle()
    n, h, w, cin, cout, k, s, dil, alpha = case
    rng = np.random.default_rng(sum(case[:8]))
    x = rng.standard_normal((n, h, w, cin)).astype(np.float32)
    wt = (rng.standard_normal((k, k, cin, cout)) / np.sqrt(k * k * cin)).astype(np.float32)
    b = rng.uniform(-0.1, 0.1, cout).astype(np.float32)
    xt = torch.tensor(x, requires_grad=True); wtt = torch.tensor(wt, requires_grad=True)
    bt = torch.tensor(b, requires_grad=True)
    ref = T.conv2d(xt, wtt, bt, stride=s, dilation=dil, alpha=None if alpha == 1.0 else alpha)
    out = ops.conv2d(cu(x), cu(wt), cu(b), s, dil, alpha)
    assert out.shape == ref.shape
    assert rel_linf(out.cpu().numpy(), ref.detach().numpy()) < 2e-5
    # backward of the linear part (dy = grad wrt pre-activation)
    pre = T.conv2d(xt, wtt, bt, stride=s, dilation=dil, alpha=None)
    g = rng.standard_normal(pre.shape).astype(np.float32)
    gx, gw, gb = torch.autograd.grad(pre, [xt, wtt, bt], grad_outputs=torch.tensor(g))
    dx = ops.conv2d_dgrad(cu(g), cu(wt), (h, w), s, dil)
    assert rel_linf(dx.cpu().numpy(), gx.numpy()) < 3e-5
    dw, db = ops.conv2d_wgrad(cu(x), cu(g), k, k, s, dil)
    assert rel_linf(dw.cpu().numpy(), gw.numpy()) < 5e-5
    assert rel_linf(db.cpu().numpy(), gb.numpy()) < 5e-5


@pytest.mark.parametrize('shape', [(1, 32, 32), (2, 37, 51), (2, 96, 160)])
def test_conv2d_stem_direct_kernels(ops, shape):
    """DispNet conv1 (7x7 stride 2, 3 -> 64) forward and filter / bias gradient on the direct CUDA-core kernels."""
    T = _oracle()
    n, h, w = shape
    rng = np.random.default_rng(sum(shape))
    x = rng.standard_normal((n, h, w, 3)).astype(np.float32)
    wt = (rng.standard_normal((7, 7, 3, 64)) / np.sqrt(147.0)).astype(np.float32)
    b = rng.uniform(-0.1, 0.1, 64).astype(np.float32)
    xt = torch.tensor(x); wtt = torch.tensor(wt, requires_grad=True); bt = torch.tensor(b, requires_grad=True)
    ref = T.conv2d(xt, wtt, bt, stride=2, dilation=1, alpha=0.1)
    out = ops.conv2d_stem(cu(x), cu(wt), cu(b), 0.1)
    assert out.shape == ref.shape
    assert rel_linf(out.cpu().numpy(), ref.detach().numpy()) < 2e-5
    pre = T.conv2d(xt, wtt, bt, stride=2, dilation=1, alpha=None)
    g = rng.standard_normal(pre.shape).astype(np.float32)
    gw, gb = torch.autograd.grad(pre, [wtt, bt], grad_outputs=torch.tensor(g))
    dw, db = ops.conv2d_stem_wgrad(cu(x), cu(g))
    assert rel_linf(dw.cpu().numpy(), gw.numpy()) < 5e-5
    assert rel_linf(db.cpu().numpy(), gb.numpy()) < 5e-5


@pytest.mark.parametrize('case', [(1, 6, 8, 32, 16, 0.1), (2, 5, 7, 1, 1, 1.0), (1, 4, 4, 64, 32, 0.1)])
def test_conv2d_transpose_fwd(ops, case):
    T = _oracle()
    n, h, w, cin, cout, alpha = case
    rng = np.random.default_rng(11)
    x = rng.standard_normal((n, h, w, cin)).astype(np.float32)
    wt = (rng.standard_normal((4, 4, cout, cin)) / 4).astype(np.float32)
    b = rng.uniform(-0.1, 0.1, cout).astype(np.float32)
    ref = T.conv2d_transpose(torch.tensor(x), torch.tensor(wt), torch.tensor(b), 2, None if alpha == 1.0 else alpha)
    out = ops.conv2d_transpose(cu(x), cu(wt), cu(b), 2, alpha)
    assert rel_linf(out.cpu().numpy(), ref.numpy()) < 2e-5


RESIZE_CASES = [
    # ih, iw, rh, rw, oh, ow, pre_scale, pre_relu, post_scale, post_relu
    (6, 20, 384, 1280, 384, 1280, -20.0, True, 1.0, False), (6, 20, 12, 40, 12, 40, 1.0, False, 0.625, False),
    (24, 32, 128, 192, 100, 180, -20.0, True, 1.0, False), (24, 32, 128, 192, 100, 180, 1.0, False, -20.0, True),
    (7, 9, 7, 9, 7, 9, 1.0, False, 2.0, False), (5, 11, 13, 17, 13, 17, 1.0, False, 1.0, False),
]


@pytest.mark.parametrize('case', RESIZE_CASES)
def test_resize_fwd_bwd(ops, case):
    T = _oracle()
    ih, iw, rh, rw, oh, ow, prs, prr, pos, por = case
    rng = np.random.default_rng(ih * iw)
    x = rng.standard_normal((2, ih, iw, 1)).astype(np.float32)
    xt = torch.tensor(x, requires_grad=True)
    v = xt * prs
    if prr: v = torch.relu(v)
    v = T.resize_bilinear(v, rh, rw) * pos
    if por: v = torch.relu(v)
    ref = T.crop_or_pad(v, oh, ow)
    out = ops.resize_bilinear(cu(x), rh, rw, oh, ow, prs, prr, pos, por)
    assert rel_linf(out.cpu().numpy(), ref.detach().numpy()) < 1e-5
    g = rng.standard_normal(ref.shape).astype(np.float32)
    (gx,) = torch.autograd.grad(ref, xt, grad_outputs=torch.tensor(g))
    dx = ops.resize_bilinear_bwd(cu(g), cu(x), rh, rw, prs, prr, pos, por)
    assert rel_linf(dx.cpu().numpy(), gx.numpy()) < 2e-5


@pytest.mark.parametrize('hw', [(40, 64), (96, 160), (37, 53)])
def test_reprojection_loss_and_gradient(ops, hw):
    T = _oracle()
    from madstereo.synthetic import make_pair
    h, w = hw
    left, right, gt = make_pair(h, w, seed=2, batch=2)
    rng = np.random.default_rng(3)
    disp = (gt + rng.normal(0, 1.5, gt.shape)).astype(np.float32)
    disp[0, 0, :4, 0] = -3.0; disp[0, 1, -3:, 0] = 500.0       # out-of-range samples hit the clamps
    dt = torch.tensor(disp, requires_grad=True)
    ref = T.reprojection_loss(dt, torch.tensor(left), torch.tensor(right))
    (gref,) = torch.autograd.grad(ref, dt)
    loss, dd = ops.reprojection_loss(cu(left), cu(right), cu(disp), with_grad=True)
    assert abs(float(loss.cpu()) - float(ref)) < 2e-6 + 1e-5 * abs(float(ref))
    assert rel_linf(dd.cpu().numpy(), gref.numpy()) < 5e-4
    loss2, none = ops.reprojection_loss(cu(left), cu(right), cu(disp), with_grad=False)
    assert none is None and float(loss2.cpu()) == float(loss.cpu())


def test_momentum_update(ops):
    T = _oracle()
    rng = np.random.default_rng(0)
    n = 100003
    w = rng.standard_normal(n).astype(np.float32); g = rng.standard_normal(n).astype(np.float32)
    m = rng.standard_normal(n).astype(np.float32)
    wr, mr = T.momentum_update(torch.tensor(w), torch.tensor(g) * 0.5, torch.tensor(m), 1e-2, 0.9)
    wc, gc, mc = cu(w)[:n], cu(g), cu(m)
    ops.momentum_update(wc, gc, mc, 1e-2, 0.9, 0.5)
    assert rel_linf(wc.cpu().numpy(), wr.numpy()) < 1e-6 and rel_linf(mc.cpu().numpy(), mr.numpy()) < 1e-6


def test_pad_reflect(ops):
    T = _oracle()
    rng = np.random.default_rng(0)
    x = rng.uniform(0, 255, (2, 100, 150, 3)).astype(np.float32)
    ref = T.pad_reflect_to_multiple(torch.tensor(x), 64)
    out = ops.pad_reflect(cu(x), 64)
    assert out.shape == ref.shape and torch.equal(out.cpu(), ref)


def test_zz_loss_factory_operator_form(ops):
    """Losses.loss_factory.get_reprojection_loss('mean_SSIM_l1') -- the reference's public entry point
    (Losses/loss_factory.py:353-395) -- on the device vs the oracle.  (Last test of the last file on purpose.)"""
    T = _oracle()
    from Losses import loss_factory
    from madstereo.synthetic import make_pair
    left, right, gt = make_pair(48, 96, seed=4, batch=1)
    disp = gt.astype(np.float32)
    ref = float(T.reprojection_loss(torch.tensor(disp), torch.tensor(left), torch.tensor(right)))
    got = loss_factory.get_reprojection_loss('mean_SSIM_l1', reduced=True)([cu(disp)], {'left': cu(left), 'right': cu(right)})
    assert abs(float(got.cpu()) - ref) < 2e-6 + 1e-5 * abs(ref)
