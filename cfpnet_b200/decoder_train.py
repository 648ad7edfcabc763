"""The decoder shell and adaptive-bins head in train mode (reference train.py:96-135 trains ``Deltar`` end to end with
autograd in fp32): ``Decoder.forward`` / ``DepthHead.forward`` dispatch here when ``self.training`` is set.

Every op is a libcfp kernel on fp32 channels-last maps.  The forward reuses the exact fp32 engine (``cfp_conv_fwd`` with
the conv bias as shift and no activation, then ``cfp_tr_bn_stats`` / ``cfp_tr_bn_apply`` / LeakyReLU for a train-mode
BatchNorm; ``cfp_upsample_concat``; ``cfp_head_bins`` / ``cfp_head_expect``; each with ``CFP_F32``).  The backward:

* a conv's input gradient is ``cfp_conv_fwd`` again, with the taps mirrored and in / out channels swapped.  That kernel
  writes 32 / 64 / 128 / 256 channels per launch, so an input gradient of 80 / 168 / 232 / 312 / 392 channels is written by
  several launches into channel slices of a buffer padded to a sum of those widths (``dgrad_slices``); the pad channels have
  zero weights and every consumer reads the buffer with its pitch;
* a conv's weight gradient is ``cfp_tr_conv_wgrad_f32`` and its bias gradient ``cfp_tr_colsum``;
* ``cfp_tr_upsample_concat_bwd_f32``, ``cfp_tr_head_expect_bwd_f32`` and ``cfp_tr_head_bins_bwd_f32`` are the adjoints of
  the resize + concat and of the head; the regressor MLP runs on ``cfp_tr_gemm`` and is recomputed from the channel mean.

Each stage is a small ``torch.autograd.Function``; plain Python composes them, so autograd stitches them to the fusion
modules' ``FusionTrainFn`` and to the histogram encoder's ``HistEncoderTrainFn``.  The pre-BatchNorm maps are kept for the
backward and the element-wise stages behind them are recomputed (as ``train.lkpm_train_bwd`` does).
"""
from __future__ import annotations

import ctypes as C
from typing import List, Tuple

import torch

from . import _lib
from . import train as T

EW_LEAKY, EW_LEAKY_GRAD = 8, 9                 # cfp_tr_ew op codes: nn.LeakyReLU() (slope 0.01) and its gradient
SERVED_WIDTHS = (256, 128, 64, 32)             # output channels the fp32 cfp_conv_fwd writes per launch


def dgrad_slices(cin: int) -> Tuple[List[Tuple[int, int]], int]:
    """Channel slices [(offset, width)] the input gradient of a conv with ``cin`` input channels is written in, and the
    padded width of the buffer: cin rounded up to 32, cut greedily into served widths (80 -> 64 + 32, 168 -> 128 + 64,
    232 -> 256, 312 -> 256 + 64, 392 -> 256 + 128 + 32)."""
    padded = (cin + 31) // 32 * 32
    out, c0 = [], 0
    while c0 < padded:
        w = next(s for s in SERVED_WIDTHS if s <= padded - c0)
        out.append((c0, w))
        c0 += w
    return out, padded


def dgrad_weights(weight: torch.Tensor):
    """conv weight [cout, cin, k, k] -> [(offset, width, w' [k*k][cout][width])] for ``conv_dgrad``: w'[t][co][ci] =
    w[k*k - 1 - t][ci][co] (taps mirrored, channels swapped), channels past cin zero."""
    cout, cin, k, _ = weight.shape
    wt = weight.detach().float().flip(2, 3).permute(2, 3, 0, 1).reshape(k * k, cout, cin)
    packs = []
    for c0, w in dgrad_slices(cin)[0]:
        n = min(w, cin - c0)
        wp = torch.zeros(k * k, cout, w, device=weight.device, dtype=torch.float32)
        wp[:, :, :n] = wt[:, :, c0:c0 + n]
        packs.append((c0, w, wp))
    return packs


def fwd_weights(weight: torch.Tensor) -> torch.Tensor:
    """conv weight [cout, cin, k, k] -> the fp32 [k*k][cin][cout] layout of cfp_conv_fwd."""
    cout, cin, k, _ = weight.shape
    return weight.detach().float().permute(2, 3, 1, 0).reshape(k * k, cin, cout).contiguous()


_zero_shift = {}


def _zeros256(dev) -> torch.Tensor:
    z = _zero_shift.get(dev)
    if z is None:
        z = _zero_shift[dev] = torch.zeros(256, device=dev, dtype=torch.float32)
    return z


def conv_fwd(x: torch.Tensor, w: torch.Tensor, shift: torch.Tensor, B: int, H: int, W: int, k: int) -> torch.Tensor:
    cin, cout = w.shape[1], w.shape[2]
    out = torch.empty(B, H, W, cout, device=x.device, dtype=torch.float32)
    _lib.call("cfp_conv_fwd", x.data_ptr(), B, H, W, cin, cout, k, 0, w.data_ptr(), shift.data_ptr(), C.c_float(1.0),
              out.data_ptr(), cout, 0, _lib.CFP_F32, _lib.stream_ptr())
    return out


def conv_dgrad(dy: torch.Tensor, weight: torch.Tensor, B: int, H: int, W: int) -> torch.Tensor:
    """Input gradient of a conv: dy [B,H,W,cout] -> [B,H,W,cin] (a view of a [B,H,W,padded] buffer; pad channels unset)."""
    cout, cin, k, _ = weight.shape
    padded = dgrad_slices(cin)[1]
    dx = torch.empty(B, H, W, padded, device=dy.device, dtype=torch.float32)
    zero = _zeros256(dy.device)
    for c0, w, wp in dgrad_weights(weight):
        _lib.call("cfp_conv_fwd", dy.data_ptr(), B, H, W, cout, w, k, 0, wp.data_ptr(), zero.data_ptr(), C.c_float(1.0),
                  dx.data_ptr(), padded, c0, _lib.CFP_F32, _lib.stream_ptr())
    return dx[..., :cin]


def wgrad_scratch_floats(B: int, H: int, W: int, cin: int, cout: int, k: int) -> int:
    return int(_lib.load().cfp_tr_conv_wgrad_scratch_floats(B, H, W, cin, cout, k))


def conv_wgrad(x: torch.Tensor, dy: torch.Tensor, B: int, H: int, W: int, k: int) -> torch.Tensor:
    """Weight gradient [cout, cin, k, k] of a conv from its input x [B,H,W,cin] and output gradient dy [B,H,W,cout]."""
    cin, cout = x.shape[-1], dy.shape[-1]
    dw = torch.empty(k * k, cin, cout, device=x.device, dtype=torch.float32)
    n = wgrad_scratch_floats(B, H, W, cin, cout, k)
    scratch = torch.empty(n, device=x.device, dtype=torch.float32) if n else None
    _lib.call("cfp_tr_conv_wgrad_f32", x.data_ptr(), dy.data_ptr(), dw.data_ptr(), _lib.ptr(scratch), B, H, W, cin, cout, k,
              _lib.stream_ptr())
    return dw.view(k, k, cin, cout).permute(3, 2, 0, 1).contiguous()


def _pitched(t: torch.Tensor) -> Tuple[torch.Tensor, int]:
    """A channels-last [B,H,W,C] gradient and its channel pitch: the padded buffer behind a ``conv_dgrad`` view is read in
    place, anything else is made contiguous."""
    B, H, W, Cc = t.shape
    p = t.stride(2)
    if t.stride(3) == 1 and p >= Cc and p % 4 == 0 and t.stride(1) == W * p and t.stride(0) == H * W * p:
        return t, p
    return t.contiguous(), Cc


def _f32_cuda(what: str, *ts):
    for t in ts:
        _lib.require_cuda(t, what)
        if t.dtype != torch.float32:
            raise _lib.CfpError(f"training runs in fp32 (as the reference trains): {what} is {t.dtype}")


def require_fp32_params(mod: torch.nn.Module) -> None:
    if any(p.dtype != torch.float32 for p in mod.parameters()):
        raise _lib.CfpError("training runs in fp32 (as the reference trains): cast the module with .float()")
    for p in mod.parameters():
        _lib.require_cuda(p, "parameter")


# ---------------------------------------------------------------------------------------------- autograd stages
class ConvFn(torch.autograd.Function):
    """conv k x k (+ bias) [-> train-mode BatchNorm -> LeakyReLU(0.01)] on a channels-last map: ``UpSampleBN``'s conv-BN-
    LeakyReLU (decoder.py:43-48) when ``bn`` is given, a plain conv (decoder.py:70,76-80, DepthRegression.conv3x3)
    otherwise.  forward(x [B,H,W,cin], bn, weight, bias[, bn.weight, bn.bias]) -> [B,H,W,cout]."""

    @staticmethod
    def forward(ctx, x, bn, weight, bias, *bn_params):
        B, H, W, _ = x.shape
        k = weight.shape[-1]
        pre = conv_fwd(x, fwd_weights(weight), T._f32c(bias), B, H, W, k)
        ctx.bn, ctx.dims = bn, (B, H, W, k)
        if bn is None:
            ctx.save_for_backward(x, weight)
            return pre
        Cc = pre.shape[-1]
        y, mean, rstd = T.bn_train_fwd(pre.view(-1, Cc), bn, relu=False)
        ctx.save_for_backward(x, weight, pre, mean, rstd)
        return T.ew(y, None, EW_LEAKY).view(pre.shape)

    @staticmethod
    def backward(ctx, dout):
        B, H, W, k = ctx.dims
        bn = ctx.bn
        with torch.cuda.device(dout.device):
            d = T._f32c(dout)
            grads_bn = ()
            if bn is None:
                x, weight = ctx.saved_tensors
                dpre = d
            else:
                x, weight, pre, mean, rstd = ctx.saved_tensors
                Cc = pre.shape[-1]
                pre2 = pre.view(-1, Cc)
                y = torch.empty_like(pre2)
                _lib.call("cfp_tr_bn_apply", pre2.data_ptr(), mean.data_ptr(), rstd.data_ptr(), T._f32c(bn.weight).data_ptr(),
                          T._f32c(bn.bias).data_ptr(), y.data_ptr(), pre2.shape[0], Cc, 0, _lib.stream_ptr())
                dy = T.ew(d.view(-1, Cc), y, EW_LEAKY_GRAD)
                dpre, dg, db = T.bn_train_bwd(dy, pre2, mean, rstd, bn, relu=False)
                dpre = dpre.view(pre.shape)
                grads_bn = (dg, db)
            cout = dpre.shape[-1]
            dbias = T.colsum(dpre.view(-1, cout))
            dw = conv_wgrad(x, dpre, B, H, W, k)
            dx = conv_dgrad(dpre, weight, B, H, W) if ctx.needs_input_grad[0] else None
        return (dx, None, dw, dbias) + grads_bn


class UpCatFn(torch.autograd.Function):
    """``UpSampleBN``'s input (decoder.py:51-58): [bilinear(align_corners) resize of lo to the skip's size | skip].
    forward(lo [B,h,w,c_lo] channels-last or None, skip [B,c_skip,H,W] NCHW) -> [B,H,W,c_lo + c_skip] channels-last.
    lo = None is the plain NCHW -> channels-last flip of the skip."""

    @staticmethod
    def forward(ctx, lo, skip):
        B, Cs, H, W = skip.shape
        if lo is None:
            h, w, c_lo, lo_p = 1, 1, 0, 0
        else:
            _, h, w, c_lo = lo.shape
            lo_p = lo.data_ptr()
        sk = T._f32c(skip)
        out = torch.empty(B, H, W, c_lo + Cs, device=skip.device, dtype=torch.float32)
        _lib.call("cfp_upsample_concat", lo_p, h, w, c_lo, max(c_lo, 4), sk.data_ptr(), Cs, out.data_ptr(), B, H, W,
                  c_lo + Cs, _lib.CFP_F32, _lib.stream_ptr())
        ctx.dims = (B, h, w, c_lo, Cs, H, W)
        return out

    @staticmethod
    def backward(ctx, dcat):
        B, h, w, c_lo, Cs, H, W = ctx.dims
        with torch.cuda.device(dcat.device):
            dcat, pitch = _pitched(dcat)
            d_lo = torch.empty(B, h, w, c_lo, device=dcat.device, dtype=torch.float32) if c_lo else None
            d_skip = torch.empty(B, Cs, H, W, device=dcat.device, dtype=torch.float32) if ctx.needs_input_grad[1] else None
            _lib.call("cfp_tr_upsample_concat_bwd_f32", dcat.data_ptr(), pitch, _lib.ptr(d_lo), h, w, c_lo, _lib.ptr(d_skip),
                      Cs if d_skip is not None else 0, B, H, W, _lib.stream_ptr())
        return d_lo, d_skip


class CatFn(torch.autograd.Function):
    """torch.cat([a, b], dim=1) of decoder.py:112,117,122 on channels-last maps (cfp_copy_channels into slices)."""

    @staticmethod
    def forward(ctx, a, b):
        B, H, W, ca = a.shape
        cb = b.shape[-1]
        out = torch.empty(B, H, W, ca + cb, device=a.device, dtype=torch.float32)
        rows = B * H * W
        st = _lib.stream_ptr()
        _lib.call("cfp_copy_channels", a.data_ptr(), ca, out.data_ptr(), ca + cb, 0, ca, rows, _lib.CFP_F32, st)
        _lib.call("cfp_copy_channels", T._f32c(b).data_ptr(), cb, out.data_ptr(), ca + cb, ca, cb, rows, _lib.CFP_F32, st)
        ctx.ca, ctx.cb = ca, cb
        return out

    @staticmethod
    def backward(ctx, d):
        ca, cb = ctx.ca, ctx.cb
        with torch.cuda.device(d.device):
            d, pitch = _pitched(d)
            B, H, W, _ = d.shape
            rows = B * H * W
            st = _lib.stream_ptr()
            da = torch.empty(B, H, W, ca, device=d.device, dtype=torch.float32)
            db = torch.empty(B, H, W, cb, device=d.device, dtype=torch.float32)
            _lib.call("cfp_copy_channels", d.data_ptr(), pitch, da.data_ptr(), ca, 0, ca, rows, _lib.CFP_F32, st)
            _lib.call("cfp_copy_channels", d.data_ptr() + 4 * ca, pitch, db.data_ptr(), cb, 0, cb, rows, _lib.CFP_F32, st)
        return da, db


class ToNchwFn(torch.autograd.Function):
    """channels-last [B,H,W,C] -> NCHW (cfp_tokens_to_nchw); the adjoint is the reverse flip."""

    @staticmethod
    def forward(ctx, x):
        B, H, W, Cc = x.shape
        return T._tokens_to_nchw(T._f32c(x), B, Cc, H, W)

    @staticmethod
    def backward(ctx, d):
        with torch.cuda.device(d.device):
            B, Cc, H, W = d.shape
            return T._nchw_to_tokens(T._f32c(d)).view(B, H, W, Cc)


class ToNhwcFn(torch.autograd.Function):
    """NCHW [B,C,H,W] -> channels-last (cfp_posenc_tokens_fwd with a zero table, as train._nchw_to_tokens)."""

    @staticmethod
    def forward(ctx, x):
        B, Cc, H, W = x.shape
        return T._nchw_to_tokens(T._f32c(x)).view(B, H, W, Cc)

    @staticmethod
    def backward(ctx, d):
        with torch.cuda.device(d.device):
            B, H, W, Cc = d.shape
            return T._tokens_to_nchw(T._f32c(d), B, Cc, H, W)


# ---------------------------------------------------------------------------------------------- the decoder shell
def decoder_train_forward(dec, img_features, hist_features, **kwargs) -> torch.Tensor:
    """``Decoder.forward`` (decoder.py:96-128) in train mode -> [B, num_classes, H/2, W/2] NCHW fp32."""
    require_fp32_params(dec)
    x0, x1, x2, x3, x4 = img_features
    _f32_cuda("img_features", x0, x1, x2, x3, x4)
    _f32_cuda("hist_features", *hist_features)
    f1, f2, f3 = hist_features
    with torch.cuda.device(x4.device):

        def conv(x, c, bn=None):
            if bn is None:
                return ConvFn.apply(x, None, c.weight, c.bias)
            return ConvFn.apply(x, bn, c.weight, c.bias, bn.weight, bn.bias)

        def up(lo, skip, mod):
            net = mod._net
            z = conv(UpCatFn.apply(lo, skip), net[0], net[1])
            return conv(z, net[3], net[4])

        def level(z, c, fusion, feat):
            d = conv(z, c)
            fused = ToNhwcFn.apply(fusion(ToNchwFn.apply(d), feat, **kwargs))
            return CatFn.apply(d, fused)

        d4 = conv(UpCatFn.apply(None, x4), dec.conv4)
        d3 = level(up(d4, x3, dec.up1), dec.conv3, dec.cross_atten3, f3)
        d2 = level(up(d3, x2, dec.up2), dec.conv2, dec.cross_atten2, f2)
        d1 = level(up(d2, x1, dec.up3), dec.conv1, dec.cross_atten1, f1)
        out = conv(up(d1, x0, dec.up4), dec.conv0)
        return ToNchwFn.apply(out)


# ---------------------------------------------------------------------------------------------- the head
class HeadFn(torch.autograd.Function):
    """``DepthRegression`` (norm 'linear') + ``conv_out`` + softmax + bin expectation (deltar.py:50-61) on a channels-last
    map: forward(head, unet [B,H,W,128], *head.parameters()) -> (bin_edges [B, n_bins + 1], pred [B,1,H,W])."""

    @staticmethod
    def forward(ctx, head, unet, *params):
        B, H, W, E = unet.shape
        dh = head.depth_head
        nb, dev, npix = head.num_classes, unet.device, H * W
        st = _lib.stream_ptr()
        ram = conv_fwd(unet, fwd_weights(dh.conv3x3.weight), T._f32c(dh.conv3x3.bias), B, H, W, 3)
        f = T._f32c
        wc = f(dh.conv1x1.weight.reshape(E, E))
        reg = dh.regressor
        mean = torch.empty(B, E, device=dev, dtype=torch.float32)
        edges = torch.empty(B, nb + 1, device=dev, dtype=torch.float32)
        centres = torch.empty(B, nb, device=dev, dtype=torch.float32)
        _lib.call("cfp_head_bins", unet.data_ptr(), E, B, npix, E, wc.data_ptr(), f(reg[0].weight).data_ptr(),
                  f(reg[0].bias).data_ptr(), f(reg[2].weight).data_ptr(), f(reg[2].bias).data_ptr(), f(reg[4].weight).data_ptr(),
                  f(reg[4].bias).data_ptr(), reg[0].weight.shape[0], nb, C.c_float(head.min_val), C.c_float(head.max_val),
                  mean.data_ptr(), edges.data_ptr(), centres.data_ptr(), _lib.CFP_F32, st)
        wout = head.conv_out[0].weight
        wout_t = wout.detach().reshape(nb, E).t().contiguous()
        pred = torch.empty(B, 1, H, W, device=dev, dtype=torch.float32)
        prob = torch.empty(B, nb, H, W, device=dev, dtype=torch.float32)
        _lib.call("cfp_head_expect", ram.data_ptr(), E, B, npix, wout_t.data_ptr(), f(head.conv_out[0].bias).data_ptr(),
                  centres.data_ptr(), nb, pred.data_ptr(), prob.data_ptr(), _lib.CFP_F32, st)
        ctx.head = head
        ctx.save_for_backward(unet, ram, mean, centres, pred, prob)
        return edges, pred

    @staticmethod
    def backward(ctx, d_edges, d_pred):
        head = ctx.head
        unet, ram, mean, centres, pred, prob = ctx.saved_tensors
        B, H, W, E = unet.shape
        nb, npix, dev = head.num_classes, H * W, unet.device
        dh, reg, f = head.depth_head, head.depth_head.regressor, T._f32c
        g = {}
        with torch.cuda.device(dev):
            st = _lib.stream_ptr()
            dpred = f(d_pred)
            dlogit = torch.empty(B * npix, nb, device=dev, dtype=torch.float32)
            dcent = torch.empty(B, nb, device=dev, dtype=torch.float32)
            scratch = torch.empty(B * ((npix + 31) // 32) * nb, device=dev, dtype=torch.float32)
            _lib.call("cfp_tr_head_expect_bwd_f32", prob.data_ptr(), pred.data_ptr(), centres.data_ptr(), dpred.data_ptr(), B, npix,
                      nb, dlogit.data_ptr(), dcent.data_ptr(), scratch.data_ptr(), st)
            # conv_out (1 x 1, 128 -> n_bins)
            co = head.conv_out[0]
            dl4 = dlogit.view(B, H, W, nb)
            g[co.bias] = T.colsum(dlogit)
            g[co.weight] = conv_wgrad(ram, dl4, B, H, W, 1)
            dram = conv_dgrad(dl4, co.weight, B, H, W).contiguous()
            # regressor, recomputed from the channel mean: conv1x1 -> Linear -> LeakyReLU -> Linear -> LeakyReLU -> Linear
            wc = f(dh.conv1x1.weight.reshape(E, E))
            r0 = T.linear_fwd(mean, wc, None)
            a0 = T.linear_fwd(r0, f(reg[0].weight), f(reg[0].bias))
            h0 = T.ew(a0, None, EW_LEAKY)
            a2 = T.linear_fwd(h0, f(reg[2].weight), f(reg[2].bias))
            h2 = T.ew(a2, None, EW_LEAKY)
            z = T.linear_fwd(h2, f(reg[4].weight), f(reg[4].bias))
            dz = torch.empty_like(z)
            _lib.call("cfp_tr_head_bins_bwd_f32", z.data_ptr(), _lib.ptr(None if d_edges is None else f(d_edges)), dcent.data_ptr(),
                      dz.data_ptr(), B, nb, C.c_float(head.min_val), C.c_float(head.max_val), st)
            g[reg[4].weight], g[reg[4].bias] = T.linear_dw(dz, h2), T.colsum(dz)
            da2 = T.ew(T.linear_dx(dz, f(reg[4].weight)), a2, EW_LEAKY_GRAD)
            g[reg[2].weight], g[reg[2].bias] = T.linear_dw(da2, h0), T.colsum(da2)
            da0 = T.ew(T.linear_dx(da2, f(reg[2].weight)), a0, EW_LEAKY_GRAD)
            g[reg[0].weight], g[reg[0].bias] = T.linear_dw(da0, r0), T.colsum(da0)
            dr0 = T.linear_dx(da0, f(reg[0].weight))
            g[dh.conv1x1.weight] = T.linear_dw(dr0, mean).view(E, E, 1, 1)
            dmean = T.linear_dx(dr0, wc).mul_(1.0 / npix)
            # conv3x3 (128 -> 128) and the channel mean's broadcast back over the pixels
            g[dh.conv3x3.bias] = T.colsum(dram.view(-1, E))
            g[dh.conv3x3.weight] = conv_wgrad(unet, dram, B, H, W, 3)
            dunet = conv_dgrad(dram, dh.conv3x3.weight, B, H, W).contiguous()
            _lib.call("cfp_tr_rowop", dunet.data_ptr(), 0, dmean.data_ptr(), dunet.data_ptr(), B * npix, E, 1, npix, T.ROW_GROUP_ADD, st)
        by_id = {id(p): t for p, t in g.items()}
        return (None, dunet) + tuple(by_id.get(id(p)) for p in head.parameters())


def head_train_forward(head, unet_out: torch.Tensor):
    """``DepthHead.forward`` in train mode: NCHW [B,128,H,W] -> (bin_edges [B, n_bins + 1], pred [B,1,H,W])."""
    require_fp32_params(head)
    _f32_cuda("unet_out", unet_out)
    with torch.cuda.device(unet_out.device):
        x = ToNhwcFn.apply(unet_out)
        return HeadFn.apply(head, x, *head.parameters())
