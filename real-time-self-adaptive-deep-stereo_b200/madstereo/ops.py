"""Operator-level Python wrappers over the C ABI (NHWC float32 CUDA tensors in, CUDA tensors out).

These mirror the reference's L1 op layer (Nets/sharedLayers.py) for eager use and for the parity tests;
the engine (csrc/engine.cu) calls the same kernels directly from C++.
"""
from ctypes import c_void_p

import torch

from ._lib import MadStereoError, check, lib


def _s():
    return c_void_p(torch.cuda.current_stream().cuda_stream)


def _p(t):
    return c_void_p(t.data_ptr()) if t is not None else c_void_p(0)


def _chk(t, name):
    if not (t.is_cuda and t.dtype == torch.float32 and t.is_contiguous()):
        raise MadStereoError('%s must be a contiguous float32 CUDA tensor' % name)


def same_out(size, stride):
    return -(-size // stride)


def correlation(x, y, max_disp, stride=1, u=None):
    """sharedLayers.correlation (Nets/sharedLayers.py:23-51); optional fused linear warp of y by u."""
    _chk(x, 'x'); _chk(y, 'y')
    b, h, w, c = x.shape
    nd = (2 * max_disp) // stride + 1
    out = torch.empty(b, h, w, nd, device=x.device, dtype=torch.float32)
    if u is not None:
        _chk(u, 'u')
    check(lib().ms_corr_fwd(_p(x), c, _p(y), c, _p(u), 1, _p(out), nd, b, h, w, c, max_disp, stride, 0, 0, _s()),
          'ms_corr_fwd')
    return out


def correlation_wide(x, y, max_disp, act_scale=64.0, out=None):
    """sharedLayers.correlation for wide windows (DispNet: max_disp = 40) on the banded tensor-core kernel
    (csrc/corr_mma.cu): fp16 hi/lo operands of x * act_scale, fp32 accumulation."""
    _chk(x, 'x'); _chk(y, 'y')
    b, h, w, c = x.shape
    nd = 2 * max_disp + 1
    if out is None:
        out = torch.empty(b, h, w, nd, device=x.device, dtype=torch.float32)
    check(lib().ms_corr_fwd_wide(_p(x), c, _p(y), c, _p(out), out.shape[-1], b, h, w, c, max_disp, float(act_scale), _s()),
          'ms_corr_fwd_wide')
    return out


def correlation_into(x, y, max_disp, out, stride=1):
    """correlation() into a pre-allocated [b,h,w,nd] tensor (no allocation inside a timed region)."""
    b, h, w, c = x.shape
    nd = (2 * max_disp) // stride + 1
    check(lib().ms_corr_fwd(_p(x), c, _p(y), c, c_void_p(0), 1, _p(out), nd, b, h, w, c, max_disp, stride, 0, 0, _s()),
          'ms_corr_fwd')
    return out


def cost_volume(x, y, max_disp, stride=1, u=None):
    """MadNet._stereo_cost_volume_correlation (+ warp, + u channel): concat([x, corr, u]) padded to 4 channels."""
    b, h, w, c = x.shape
    nd = (2 * max_disp) // stride + 1
    ct = c + nd + (1 if u is not None else 0)
    cs = (ct + 3) // 4 * 4
    out = torch.zeros(b, h, w, cs, device=x.device, dtype=torch.float32)
    if u is not None:
        out[..., c + nd] = u[..., 0]
    up = c_void_p(out.data_ptr() + 4 * (c + nd)) if u is not None else c_void_p(0)
    check(lib().ms_corr_fwd(_p(x), c, _p(y), c, up, cs, _p(out), cs, b, h, w, c, max_disp, stride, 1,
                            1 if u is not None else 0, _s()), 'ms_corr_fwd')
    return out[..., :ct]


def correlation_bwd(x, y, dcorr, max_disp, stride=1, u=None, want_du=False):
    """Gradient of correlation (and warp) wrt x, y (and u)."""
    b, h, w, c = x.shape
    nd = (2 * max_disp) // stride + 1
    cs = (c + nd + 3) // 4 * 4
    dcost = torch.zeros(b, h, w, cs, device=x.device, dtype=torch.float32)
    dcost[..., c:c + nd] = dcorr
    dx = torch.empty_like(x)
    dy = torch.empty_like(y)
    du = torch.empty(b, h, w, 1, device=x.device, dtype=torch.float32) if (want_du and u is not None) else None
    check(lib().ms_corr_bwd(_p(x), c, _p(y), c, _p(u), 1, _p(dcost), cs, _p(dx), c, _p(dy), c, _p(du), 1,
                            b, h, w, c, max_disp, stride, 0, _s()), 'ms_corr_bwd')
    return dx, dy, du


def conv2d(x, w, b, stride=1, dilation=1, alpha=1.0):
    """sharedLayers.conv2d / dilated_conv2d (Nets/sharedLayers.py:54-77). w HWIO."""
    _chk(x, 'x'); _chk(w, 'w')
    n, h, wd, cin = x.shape
    kh, kw, _, cout = w.shape
    y = torch.empty(n, same_out(h, stride), same_out(wd, stride), cout, device=x.device, dtype=torch.float32)
    check(lib().ms_conv2d_fwd(_p(x), n, h, wd, cin, cin, _p(w), _p(b), _p(y), cout, cout, kh, kw, stride, dilation,
                              float(alpha), _s()), 'ms_conv2d_fwd')
    return y


def conv2d_bf(x, w, b, stride=1, dilation=1, alpha=1.0, act_scale=0.0625):
    """split-bf16 tcgen05 forward conv (csrc/conv_bf.cu; same semantics as conv2d, stride 1 or 2)."""
    n, h, wd, cin = x.shape
    kh, kw, _, cout = w.shape
    y = torch.empty(n, same_out(h, stride), same_out(wd, stride), cout, device=x.device, dtype=torch.float32)
    ns = lib().ms_conv2d_bf_scratch(n, h, wd, kh, kw, cin, cout)
    scratch = torch.empty(ns + 256, device=x.device, dtype=torch.uint8)
    off = (-scratch.data_ptr()) % 256
    check(lib().ms_conv2d_fwd_bf(_p(x), n, h, wd, cin, cin, _p(w), _p(b), _p(y), cout, cout, kh, kw, stride, dilation,
                                 float(alpha), float(act_scale), c_void_p(scratch.data_ptr() + off), ns, _s()), 'ms_conv2d_fwd_bf')
    return y


def conv2d_dgrad_bf(dy, w, in_hw=None, stride=1, dilation=1):
    n, oh, ow, cout = dy.shape
    kh, kw, cin, _ = w.shape
    h, wd = in_hw if in_hw is not None else (oh, ow)
    dx = torch.empty(n, h, wd, cin, device=dy.device, dtype=torch.float32)
    ns = lib().ms_conv2d_bf_scratch(n, h, wd, kh, kw, cin, cout)
    scratch = torch.empty(ns + 256, device=dy.device, dtype=torch.uint8)
    off = (-scratch.data_ptr()) % 256
    check(lib().ms_conv2d_dgrad_bf(_p(dy), n, oh, ow, cout, cout, _p(w), _p(dx), h, wd, cin, cin, kh, kw, stride, dilation,
                                   c_void_p(scratch.data_ptr() + off), ns, _s()), 'ms_conv2d_dgrad_bf')
    return dx


def conv2d_wgrad_bf(x, dy, kh, kw, stride=1, dilation=1):
    """tcgen05 weight + bias gradient on bf16 hi/lo planes (csrc/wgrad_bf.cu), stride 1 or 2."""
    n, h, wd, cin = x.shape
    _, oh, ow, cout = dy.shape
    dw = torch.empty(kh, kw, cin, cout, device=x.device, dtype=torch.float32)
    db = torch.empty(cout, device=x.device, dtype=torch.float32)
    ns = lib().ms_conv2d_wgrad_bf_scratch(n, h, wd, oh, ow, kh, kw, cin, cout)
    scratch = torch.empty(ns + 256, device=x.device, dtype=torch.uint8)
    off = (-scratch.data_ptr()) % 256
    check(lib().ms_conv2d_wgrad_bf(_p(x), n, h, wd, cin, cin, _p(dy), oh, ow, cout, cout, _p(dw), _p(db), kh, kw, stride,
                                   dilation, c_void_p(scratch.data_ptr() + off), ns, _s()), 'ms_conv2d_wgrad_bf')
    return dw, db


def _pad4(x):
    n, h, w, c = x.shape
    x4 = torch.zeros(n, h, w, 4, device=x.device, dtype=torch.float32)
    x4[..., :c] = x
    return x4


def conv2d_stem(x, w, b, alpha=0.1):
    """DispNet conv1 (7x7 stride 2, 3 -> 64) on the direct kernel (csrc/conv_stem.cu). x [n,h,w,3]."""
    n, h, wd, _ = x.shape
    y = torch.empty(n, same_out(h, 2), same_out(wd, 2), 64, device=x.device, dtype=torch.float32)
    x4 = _pad4(x)
    check(lib().ms_conv2d_stem_fwd(_p(x4), n, h, wd, _p(w), _p(b), _p(y), 64, float(alpha), _s()), 'ms_conv2d_stem_fwd')
    return y


def conv2d_stem_wgrad(x, dy):
    n, h, wd, _ = x.shape
    dw = torch.empty(7, 7, 3, 64, device=x.device, dtype=torch.float32)
    db = torch.empty(64, device=x.device, dtype=torch.float32)
    nws = lib().ms_conv2d_stem_wgrad_workspace(n, h, wd)
    ws = torch.empty(nws, device=x.device, dtype=torch.float32)
    x4 = _pad4(x)
    check(lib().ms_conv2d_stem_wgrad(_p(x4), n, h, wd, _p(dy), 64, _p(dw), _p(db), _p(ws), nws, _s()), 'ms_conv2d_stem_wgrad')
    return dw, db


def _scratch256(nbytes, device):
    buf = torch.empty(nbytes + 256, device=device, dtype=torch.uint8)
    return buf, c_void_p(buf.data_ptr() + (-buf.data_ptr()) % 256)


def conv2d_transpose_bf(x, w, b, stride=2, alpha=1.0, act_scale=0.0625):
    """sharedLayers.conv2d_transpose on the tcgen05 path (fp16 hi/lo planes). w [kh,kw,cout,cin]."""
    n, h, wd, cin = x.shape
    kh, kw, cout, _ = w.shape
    y = torch.empty(n, h * stride, wd * stride, cout, device=x.device, dtype=torch.float32)
    ns = lib().ms_conv2d_transpose_bf_scratch(n, h, wd, kh, kw, cin, cout, stride)
    keep, sp = _scratch256(ns, x.device)
    check(lib().ms_conv2d_transpose_fwd_bf(_p(x), n, h, wd, cin, cin, _p(w), _p(b), _p(y), cout, cout, kh, kw, stride,
                                           float(alpha), float(act_scale), sp, ns, _s()), 'ms_conv2d_transpose_fwd_bf')
    return y


def conv2d_transpose_dgrad_bf(dy, w, stride=2):
    """d(conv2d_transpose)/dx on the tcgen05 path (bf16 hi/lo planes). dy [n,h*s,w*s,cout], w [kh,kw,cout,cin]."""
    n, oh, ow, cout = dy.shape
    kh, kw, _, cin = w.shape
    h, wd = oh // stride, ow // stride
    dx = torch.empty(n, h, wd, cin, device=dy.device, dtype=torch.float32)
    ns = lib().ms_conv2d_transpose_bf_scratch(n, h, wd, kh, kw, cin, cout, stride)
    keep, sp = _scratch256(ns, dy.device)
    check(lib().ms_conv2d_transpose_dgrad_bf(_p(dy), n, h, wd, cout, cout, _p(w), _p(dx), cin, cin, kh, kw, stride, sp, ns,
                                             _s()), 'ms_conv2d_transpose_dgrad_bf')
    return dx


def conv2d_transpose_wgrad_bf(x, dy, kh, kw, stride=2):
    """d(conv2d_transpose)/dW [kh,kw,cout,cin] and /db [cout] on the tcgen05 path (bf16 hi/lo planes)."""
    n, h, wd, cin = x.shape
    cout = dy.shape[3]
    dw = torch.empty(kh, kw, cout, cin, device=x.device, dtype=torch.float32)
    db = torch.empty(cout, device=x.device, dtype=torch.float32)
    ns = lib().ms_conv2d_transpose_wgrad_bf_scratch(n, h, wd, kh, kw, cin, cout, stride)
    keep, sp = _scratch256(ns, x.device)
    check(lib().ms_conv2d_transpose_wgrad_bf(_p(x), n, h, wd, cin, cin, _p(dy), cout, cout, _p(dw), _p(db), kh, kw, stride,
                                             sp, ns, _s()), 'ms_conv2d_transpose_wgrad_bf')
    return dw, db


def conv2d_dgrad(dy, w, in_hw, stride=1, dilation=1):
    n, oh, ow, cout = dy.shape
    kh, kw, cin, _ = w.shape
    h, wd = in_hw
    dx = torch.empty(n, h, wd, cin, device=dy.device, dtype=torch.float32)
    scratch = torch.empty(w.numel(), device=dy.device, dtype=torch.float32)
    check(lib().ms_conv2d_dgrad(_p(dy), n, oh, ow, cout, cout, _p(w), _p(dx), h, wd, cin, cin, kh, kw, stride,
                                dilation, _p(scratch), _s()), 'ms_conv2d_dgrad')
    return dx


def conv2d_wgrad(x, dy, kh, kw, stride=1, dilation=1):
    n, h, wd, cin = x.shape
    _, oh, ow, cout = dy.shape
    dw = torch.empty(kh, kw, cin, cout, device=x.device, dtype=torch.float32)
    db = torch.empty(cout, device=x.device, dtype=torch.float32)
    nws = lib().ms_conv2d_wgrad_workspace(kh, kw, cin, cout, n * oh * ow)
    ws = torch.empty(nws, device=x.device, dtype=torch.float32)
    check(lib().ms_conv2d_wgrad(_p(x), n, h, wd, cin, cin, _p(dy), oh, ow, cout, cout, _p(dw), _p(db), kh, kw,
                                stride, dilation, _p(ws), nws, _s()), 'ms_conv2d_wgrad')
    return dw, db


def conv2d_wgrad_tc(x, dy, kh, kw, dilation=1):
    """tcgen05 / 3xTF32 weight + bias gradient of a stride-1 conv."""
    n, h, wd, cin = x.shape
    cout = dy.shape[3]
    dw = torch.empty(kh, kw, cin, cout, device=x.device, dtype=torch.float32)
    db = torch.empty(cout, device=x.device, dtype=torch.float32)
    nws = lib().ms_conv2d_wgrad_tc_workspace(kh, kw, cin, cout, n, h, wd)
    ws = torch.empty(nws, device=x.device, dtype=torch.float32)
    check(lib().ms_conv2d_wgrad_tc(_p(x), n, h, wd, cin, cin, _p(dy), cout, cout, _p(dw), _p(db), kh, kw, dilation,
                                   _p(ws), nws, _s()), 'ms_conv2d_wgrad_tc')
    return dw, db


def conv2d_transpose(x, w, b, stride=2, alpha=1.0):
    """sharedLayers.conv2d_transpose (Nets/sharedLayers.py:80-92). w [kh,kw,cout,cin]."""
    n, h, wd, cin = x.shape
    kh, kw, cout, _ = w.shape
    y = torch.empty(n, h * stride, wd * stride, cout, device=x.device, dtype=torch.float32)
    scratch = torch.empty(w.numel(), device=x.device, dtype=torch.float32)
    check(lib().ms_conv2d_transpose_fwd(_p(x), n, h, wd, cin, cin, _p(w), _p(b), _p(y), cout, cout, kh, kw, stride,
                                        float(alpha), _p(scratch), _s()), 'ms_conv2d_transpose_fwd')
    return y


def resize_bilinear(x, rh, rw, oh=None, ow=None, pre_scale=1.0, pre_relu=False, post_scale=1.0, post_relu=False):
    oh = rh if oh is None else oh
    ow = rw if ow is None else ow
    b, ih, iw, c = x.shape
    assert c == 1
    y = torch.empty(b, oh, ow, 1, device=x.device, dtype=torch.float32)
    check(lib().ms_resize_bilinear(_p(x), 1, b, ih, iw, _p(y), 1, rh, rw, oh, ow, pre_scale, int(pre_relu),
                                   post_scale, int(post_relu), _s()), 'ms_resize_bilinear')
    return y


def resize_bilinear_bwd(dout, x, rh, rw, pre_scale=1.0, pre_relu=False, post_scale=1.0, post_relu=False):
    b, ih, iw, _ = x.shape
    _, oh, ow, _ = dout.shape
    dx = torch.empty_like(x)
    tmp = torch.empty(b * oh * iw, device=x.device, dtype=torch.float32)
    check(lib().ms_resize_bilinear_bwd(_p(dout), 1, _p(x), 1, b, ih, iw, _p(dx), 1, rh, rw, oh, ow, pre_scale,
                                       int(pre_relu), post_scale, int(post_relu), 0, _p(tmp), _s()),
          'ms_resize_bilinear_bwd')
    return dx


def reprojection_loss(left, right, disp, with_grad=False):
    """loss_factory.get_reprojection_loss('mean_SSIM_l1') (Losses/loss_factory.py:353-395). Returns (loss, ddisp)."""
    b, h, w, _ = left.shape
    ws = torch.empty(lib().ms_reproj_loss_workspace(b, h, w), device=left.device, dtype=torch.float32)
    loss = torch.zeros(1, device=left.device, dtype=torch.float32)
    dd = torch.empty(b, h, w, 1, device=left.device, dtype=torch.float32) if with_grad else None
    check(lib().ms_reproj_loss(_p(left), _p(right), _p(disp), b, h, w, _p(loss), _p(dd), _p(ws), 1.0, _s()),
          'ms_reproj_loss')
    return loss, dd


def momentum_update(w, g, m, lr, mu=0.9, grad_scale=1.0):
    check(lib().ms_momentum_update(_p(w), _p(g), _p(m), w.numel(), lr, mu, grad_scale, _s()), 'ms_momentum_update')


def pad_reflect(x, factor=64, scale=1.0, bias=0.0):
    b, h, w, c = x.shape
    hp, wp = -(-h // factor) * factor, -(-w // factor) * factor
    y = torch.empty(b, hp, wp, c, device=x.device, dtype=torch.float32)
    check(lib().ms_pad_reflect(_p(x), b, h, w, c, _p(y), hp, wp, c, scale, bias, _s()), 'ms_pad_reflect')
    return y
