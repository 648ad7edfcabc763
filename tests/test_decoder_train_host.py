"""CPU checks of the decoder shell / head training path's host arithmetic: the input-gradient weight packing and channel-slice
plan (applied by a restatement of what the fp32 cfp_conv_fwd computes per tap) against torch's conv2d_input, the gather ranges
and weights of the upsample adjoint (restated in fp32 as cfp_tr_upsample_concat_bwd_f32 forms them) against autograd of
F.interpolate, the train-mode fp64 reference of UpSampleBN the GPU tests compare against, and the weight-gradient scratch
size (pure host arithmetic).  No device work."""
import math

import numpy as np
import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

from cfpnet_b200 import _lib, decoder as D
from cfpnet_b200 import decoder_train as DT
from oracle import cfp_oracle as O

# (cin, cout, k) of every conv of the decoder shell (decoder.py:70-80, 43-48, num_classes 128) and of the head
# (DepthRegression.conv3x3, conv_out)
CONV_SHAPES = [(232, 256, 1), (392, 256, 3), (256, 256, 3), (256, 128, 1), (312, 128, 3), (128, 128, 3), (128, 64, 1),
               (168, 64, 3), (64, 64, 3), (64, 32, 1), (80, 32, 3), (32, 32, 3), (32, 128, 3), (128, 128, 3), (128, 256, 1)]


def conv_f32_restated(x_nhwc, w, out, out_coff):
    """What the fp32 cfp_conv_fwd computes (zero shift, slope 1): out[..., coff + o] = sum_{tap, c} x[p + off(tap)][c] w[tap][c][o]."""
    B, H, W, _ = x_nhwc.shape
    taps, _, n = w.shape
    k = int(round(math.sqrt(taps)))
    xp = F.pad(x_nhwc, (0, 0, k // 2, k // 2, k // 2, k // 2))
    acc = torch.zeros(B, H, W, n, dtype=x_nhwc.dtype)
    for t in range(taps):
        dy, dx = t // k, t % k
        acc += xp[:, dy:dy + H, dx:dx + W, :] @ w[t].to(x_nhwc.dtype)
    out[..., out_coff:out_coff + n] = acc


@pytest.mark.parametrize("cin,cout,k", CONV_SHAPES)
def test_dgrad_packing_and_slices_give_the_input_gradient(cin, cout, k):
    g = torch.Generator().manual_seed(cin * 7 + cout + k)
    B, H, W = 2, 5, 7
    weight = torch.randn(cout, cin, k, k, generator=g, dtype=torch.float64)
    dy = torch.randn(B, cout, H, W, generator=g, dtype=torch.float64)
    slices, padded = DT.dgrad_slices(cin)
    assert all(w in (32, 64, 128, 256) for _, w in slices)
    assert sum(w for _, w in slices) == padded >= cin and padded - cin < 32
    assert [c0 for c0, _ in slices] == [sum(w for _, w in slices[:i]) for i in range(len(slices))]
    packs = DT.dgrad_weights(weight)
    out = torch.full((B, H, W, padded), float("nan"), dtype=torch.float64)
    for c0, w, wp in packs:
        assert wp.shape == (k * k, cout, w) and wp.dtype == torch.float32
        assert (wp[:, :, max(0, cin - c0):] == 0).all(), "pad channels must have zero weights"
        conv_f32_restated(dy.permute(0, 2, 3, 1), wp.double(), out, c0)
    want = torch.nn.grad.conv2d_input((B, cin, H, W), weight.float().double(), dy, padding=k // 2)
    got = out[..., :cin].permute(0, 3, 1, 2)
    assert torch.allclose(got, want, rtol=1e-12, atol=1e-12)


def test_dgrad_slice_plan_of_the_decoder_widths():
    plan = {c: [w for _, w in DT.dgrad_slices(c)[0]] for c in (80, 168, 232, 312, 392, 32, 64, 128, 256)}
    assert plan == {80: [64, 32], 168: [128, 64], 232: [256], 312: [256, 64], 392: [256, 128, 32],
                    32: [32], 64: [64], 128: [128], 256: [256]}


# ---------------------------------------------------------------------------------------------- upsample adjoint
f32 = np.float32


def _interp_weight(y, j, s, n):
    fy = f32(s * f32(y))
    y0 = min(int(fy), n - 1)
    y1 = y0 + (1 if y0 < n - 1 else 0)
    l_ = f32(fy - f32(y0))
    return (f32(1) - l_ if y0 == j else f32(0)) + (l_ if y1 == j else f32(0))


def _gather_range(j, s, N):
    if not s > 0:
        return 0, N - 1
    a = min(f32(f32(j - 1) / s), f32(N))
    b = min(f32(f32(j + 1) / s), f32(N))
    return max(0, math.floor(a) - 1), min(N - 1, math.ceil(b) + 1)


def _adjoint_matrix(n, N, gather=True):
    """A[j, y]: weight with which destination row y feeds source row j, over the rows the kernel's gather visits
    (``gather``) or over every row."""
    s = f32(f32(n - 1) / f32(N - 1)) if N > 1 else f32(0)
    A = np.zeros((n, N))
    for j in range(n):
        lo, hi = _gather_range(j, s, N) if gather else (0, N - 1)
        for y in range(lo, hi + 1):
            A[j, y] = _interp_weight(y, j, s, n)
    return A


def _levels(img_h, img_w):
    return [((img_h // a, img_w // a), (img_h // b, img_w // b)) for a, b in ((32, 32), (32, 16), (16, 8), (8, 4), (4, 2))]


@pytest.mark.parametrize("lo,hi", _levels(416, 544) + _levels(480, 640) + [((7, 5), (23, 9)), ((1, 3), (4, 8))])
def test_upsample_adjoint_gather_matches_autograd(lo, hi):
    (h, w), (H, W) = lo, hi
    g = torch.Generator().manual_seed(h * 1000 + W)
    x = torch.randn(1, 2, h, w, dtype=torch.float64, requires_grad=True)
    dout = torch.randn(1, 2, H, W, generator=g, dtype=torch.float64)
    F.interpolate(x, size=[H, W], mode="bilinear", align_corners=True).backward(dout)
    Ay, Ax = _adjoint_matrix(h, H), _adjoint_matrix(w, W)
    # the gather visits every destination row / column with a non-zero weight
    assert np.array_equal(Ay, _adjoint_matrix(h, H, gather=False)) and np.array_equal(Ax, _adjoint_matrix(w, W, gather=False))
    got = torch.einsum("jy,bcyx,ix->bcji", torch.from_numpy(Ay), dout, torch.from_numpy(Ax))
    # the source coordinates are formed in fp32 as in the forward kernel (error ~ coordinate x 6e-8), autograd's in fp64
    err = float((got - x.grad).norm() / x.grad.norm())
    assert err <= 1e-5, err


# ---------------------------------------------------------------------------------------------- train-mode fp64 reference
def upsample_bn_train(p, x, concat_with, bn_stats):
    """``UpSampleBN.forward`` (decoder.py:40-58) in train mode: the oracle's ``upsample_bn`` with batch-statistics BatchNorm
    (``O._bn`` with a ``bn_stats`` dict records the updated running buffers)."""
    up = F.interpolate(x, size=[concat_with.size(2), concat_with.size(3)], mode="bilinear", align_corners=True)
    f = torch.cat([up, concat_with], dim=1)
    f = F.leaky_relu(O._bn(O._conv(p, "_net.0", f, 1), p, "_net.1", 1, bn_stats), 0.01)
    return F.leaky_relu(O._bn(O._conv(p, "_net.3", f, 1), p, "_net.4", 1, bn_stats), 0.01)


def decoder_shell_train(p, img_features, hist_features, fuse, bn_stats):
    """``Decoder.forward`` (decoder.py:96-128) in train mode, as ``O.decoder_shell`` with ``upsample_bn_train``."""
    x0, x1, x2, x3, x4 = img_features
    f1, f2, f3 = hist_features
    d4 = O._conv(p, "conv4", x4, 0)
    d3 = O._conv(p, "conv3", upsample_bn_train(O.sub(p, "up1."), d4, x3, bn_stats), 0)
    d3 = torch.cat([d3, fuse("cross_atten3", d3, f3)], dim=1)
    d2 = O._conv(p, "conv2", upsample_bn_train(O.sub(p, "up2."), d3, x2, bn_stats), 0)
    d2 = torch.cat([d2, fuse("cross_atten2", d2, f2)], dim=1)
    d1 = O._conv(p, "conv1", upsample_bn_train(O.sub(p, "up3."), d2, x1, bn_stats), 0)
    d1 = torch.cat([d1, fuse("cross_atten1", d1, f1)], dim=1)
    d0 = upsample_bn_train(O.sub(p, "up4."), d1, x0, bn_stats)
    return O._conv(p, "conv0", d0, 1)


def test_train_mode_upsample_bn_reference_matches_the_module():
    torch.manual_seed(0)
    mod = D.UpSampleBN(24 + 8, 16).double()
    for bn in (mod._net[1], mod._net[4]):
        with torch.no_grad():
            bn.weight.uniform_(0.5, 1.5)
            bn.bias.normal_(0, 0.2)
            bn.running_mean.normal_(0, 0.2)
            bn.running_var.uniform_(0.5, 1.5)
    sd = {k: v.clone() for k, v in mod.state_dict().items()}
    x = torch.randn(2, 24, 5, 6, dtype=torch.float64)
    skip = torch.randn(2, 8, 9, 11, dtype=torch.float64)
    stats = {}
    got = upsample_bn_train(O.sub({"up1." + k: v for k, v in sd.items()}, "up1."), x, skip, stats)
    mod.train()
    up = F.interpolate(x, size=[9, 11], mode="bilinear", align_corners=True)
    want = mod._net(torch.cat([up, skip], dim=1))
    assert torch.allclose(got, want, rtol=1e-12, atol=1e-12)
    after = mod.state_dict()
    assert sorted(stats) == sorted("up1." + k for k in after if "running" in k or "num_batches" in k)
    for k, v in stats.items():
        ref = after[k[len("up1."):]]
        assert torch.equal(v, ref) if ref.dtype == torch.int64 else torch.allclose(v, ref, rtol=1e-12, atol=1e-14), k


# ---------------------------------------------------------------------------------------------- wgrad scratch
@pytest.fixture(scope="module")
def lib():
    from cfpnet_b200.build import build
    build()
    return _lib.load()


def _splits(K, cin, cout, taps):
    """Restatement of the pixel-range split of csrc/k_dec_train.cu (wg::plan)."""
    tiles = -(-cin // 64) * -(-cout // 64) * taps
    s = max(1, min(-(-1184 // tiles), -(-K // 512)))
    kchunk = -(-(-(-K // s)) // 32) * 32
    return -(-K // kchunk)


@pytest.mark.parametrize("B,H,W,cin,cout,k", [(16, 208, 272, 32, 32, 3), (16, 13, 17, 392, 256, 3), (16, 208, 272, 128, 256, 1),
                                              (1, 45, 37, 80, 32, 3), (2, 4, 4, 64, 64, 1), (1, 1, 1, 4, 4, 3)])
def test_wgrad_scratch_size_is_pure_host_arithmetic(lib, B, H, W, cin, cout, k):
    n = lib.cfp_tr_conv_wgrad_scratch_floats(B, H, W, cin, cout, k)
    s = _splits(B * H * W, cin, cout, k * k)
    assert n == (s * k * k * cin * cout if s > 1 else 0)
    assert n == DT.wgrad_scratch_floats(B, H, W, cin, cout, k)
    assert lib.cfp_tr_conv_wgrad_scratch_floats(B, H, W, cin, cout, 5) == 0
    assert lib.cfp_tr_conv_wgrad_scratch_floats(0, H, W, cin, cout, k) == 0
