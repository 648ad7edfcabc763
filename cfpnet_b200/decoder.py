"""Decoder shell and adaptive-bins head around the fusion path (SURVEY.md 8 f1 / f2): bf16 on the tensor cores, or the exact
fp32 engine (``Decoder.compute_dtype = torch.float32``; the head follows the dtype of the map it is given).

Mirrors ``src/models/decoder.py`` (``UpSampleBN``, ``Decoder``, ``DepthRegression``) and the head wiring of
``src/models/deltar.py:15-19,50-61``: same constructor arguments, same ``state_dict`` keys and shapes, so a reference
checkpoint loads with ``strict=True``.  The maps stay channels-last bf16 between the kernels (the token-major layout of
the fusion layers): every ``torch.cat`` of the reference is a write into a slice of a wider buffer, the bilinear
upsample + skip concat is one kernel, convs are ``cfp_conv_fwd`` (tcgen05 implicit GEMM with the eval-mode BatchNorm folded
and LeakyReLU in the epilogue), and ``conv_out`` + softmax + bin expectation is ``cfp_head_expect`` (the 256-bin
probability volume is only written on request).  The fp32 engine runs the same sequence on fp32 maps through
the ``*_f32`` kernels (FFMA, fixed summation order) and the fusion modules' fp32 engine.  Eval mode only; no CPU fallback.
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, List, Tuple

import torch
import torch.nn as nn

from . import _lib
from .fusion import TransformerFusion
from .packing import PackCache, fold_bn, host, umma_block


def _pad16(c: int) -> int:
    return (c + 15) // 16 * 16


def _conv_plan(cin: int, cout: int, may_pad: bool) -> Tuple[int, int]:
    """(cin_pad, kc) for ``cfp_conv_fwd``: input channels padded to a multiple of 16 and the K-chunk kc (channels staged per
    pass): the largest multiple of 16 dividing cin_pad whose weight block fits a 40 KB ring slot and whose two raster
    buffers + ring fit 200 KB of shared memory (the launcher's formula, csrc/k_dec_tc.cu: conv_gen_launch).  When the
    input is a buffer this module lays out itself (``may_pad``), up to 48 extra zero channels are allowed if they cut the
    number of chunks (176 = 11 x 16 channels would run as 11 chunks, 192 as 3)."""
    cap = (2 if cout >= 128 else 4) * 128
    cells = cap + 2 * ((34 if cap == 256 else 46) + 2) + 2 + 8

    def best_kc(cp):
        best, m = 16, cp // 16
        for d in range(1, m + 1):
            kc = 16 * d
            if m % d == 0 and cout * kc <= 20480 and 2 * (kc // 8) * cells * 16 + 2 * cout * kc * 2 <= 200 * 1024:
                best = kc
        return best

    base = _pad16(cin)
    cands = [base + 16 * i for i in range(4)] if may_pad else [base]
    cp = min(cands, key=lambda c: (c // best_kc(c), c))
    return cp, best_kc(cp)


class _PackedConv:
    """One conv (+ folded BatchNorm) packed for cfp_conv_fwd: bf16 blocks [chunk][tap][kc/8][cout][8] + fp32 shift; with
    ``dtype=torch.float32`` for cfp_conv_f32_fwd: fp32 [tap][cin][cout], input channels not padded."""

    def __init__(self, conv: nn.Conv2d, bn: nn.BatchNorm2d | None, device, may_pad: bool = False, dtype=torch.bfloat16):
        w = host(conv.weight)                                              # [cout, cin, k, k]
        cout, cin, k, _ = w.shape
        if bn is not None:
            scale, shift = fold_bn(bn)
            w = w * scale[:, None, None, None]
            if conv.bias is not None:
                shift = shift + host(conv.bias) * scale
        else:
            shift = host(conv.bias) if conv.bias is not None else torch.zeros(cout)
        self.cin, self.cout, self.k, self.dtype = cin, cout, k, dtype
        self.shift = shift.float().contiguous().to(device)
        if dtype == torch.float32:
            self.cin_pad, self.kc = cin, 0
            self.w = w.permute(2, 3, 1, 0).reshape(k * k, cin, cout).contiguous().to(device)
            return
        self.cin_pad, self.kc = _conv_plan(cin, cout, may_pad)
        wp = torch.zeros(cout, self.cin_pad, k, k)
        wp[:, :cin] = w
        blocks = [umma_block(wp[:, c0:c0 + self.kc, ky, kx]) for c0 in range(0, self.cin_pad, self.kc)
                  for ky in range(k) for kx in range(k)]
        self.w_tc = torch.stack(blocks).contiguous().to(device)


class UpSampleBN(nn.Module):
    """decoder.py:40-58 (parameters only; the forward is sequenced by ``Decoder``)."""

    def __init__(self, skip_input, output_features):
        super().__init__()
        self._net = nn.Sequential(nn.Conv2d(skip_input, output_features, kernel_size=3, stride=1, padding=1),
                                  nn.BatchNorm2d(output_features), nn.LeakyReLU(),
                                  nn.Conv2d(output_features, output_features, kernel_size=3, stride=1, padding=1),
                                  nn.BatchNorm2d(output_features), nn.LeakyReLU())


def _conv(pc: _PackedConv, x: torch.Tensor, B: int, H: int, W: int, slope: float, out: torch.Tensor, out_pitch: int, out_coff: int):
    if pc.dtype == torch.float32:
        _lib.call("cfp_conv_f32_fwd", x.data_ptr(), B, H, W, pc.cin, pc.cout, pc.k, pc.w.data_ptr(), pc.shift.data_ptr(),
                  C.c_float(slope), out.data_ptr(), out_pitch, out_coff, _lib.stream_ptr())
        return
    _lib.call("cfp_conv_fwd", x.data_ptr(), B, H, W, pc.cin_pad, pc.cout, pc.k, pc.kc, pc.w_tc.data_ptr(), pc.shift.data_ptr(),
              C.c_float(slope), out.data_ptr(), out_pitch, out_coff, _lib.stream_ptr())


class Decoder(nn.Module):
    """decoder.py:60-128.  ``forward(img_features, hist_features, **kwargs)`` returns the reference's ``[B, num_classes,
    h/2, w/2]`` map (NCHW, fp32); ``forward_nhwc`` returns it channels-last in ``compute_dtype`` for ``DepthHead``.

    ``compute_dtype`` selects the engine: ``torch.bfloat16`` (default) runs the tcgen05 kernels with bf16 maps and the
    fusion modules in whatever dtype they were cast to (bf16 for the tensor-core engine); ``torch.float32`` runs the
    exact fp32 kernels on fp32 maps and needs the ``cross_atten*`` modules left in fp32 (their fp32 engine)."""

    LEAKY = 0.01                                  # nn.LeakyReLU() default

    def __init__(self, num_classes=1):
        super().__init__()
        if num_classes not in (32, 64, 128, 256):
            raise NotImplementedError("libcfp serves conv0 with 32 / 64 / 128 / 256 output channels (deltar.py:17 uses 128)")
        encoder_channels = [232, 136, 56, 40, 16]
        decoder_channels = [256, 256, 128, 64, 32]
        self.conv4 = nn.Conv2d(encoder_channels[0], decoder_channels[0], kernel_size=1, stride=1, padding=0)
        self.up1 = UpSampleBN(decoder_channels[0] + encoder_channels[1], decoder_channels[1])
        self.up2 = UpSampleBN(decoder_channels[1] + encoder_channels[2], decoder_channels[2])
        self.up3 = UpSampleBN(decoder_channels[2] + encoder_channels[3], decoder_channels[3])
        self.up4 = UpSampleBN(decoder_channels[3] + encoder_channels[4], decoder_channels[4])
        self.conv3 = nn.Conv2d(decoder_channels[1], decoder_channels[2], kernel_size=1, stride=1, padding=0)
        self.conv2 = nn.Conv2d(decoder_channels[2], decoder_channels[3], kernel_size=1, stride=1, padding=0)
        self.conv1 = nn.Conv2d(decoder_channels[3], decoder_channels[4], kernel_size=1, stride=1, padding=0)
        self.conv0 = nn.Conv2d(decoder_channels[4], num_classes, kernel_size=3, stride=1, padding=1)
        resolution = [[240, 320], [120, 160], [60, 80], [30, 40], [15, 20]]
        channels = [int(c / 2) for c in decoder_channels]
        self.cross_atten1 = TransformerFusion(embedding_dim=channels[3], max_resolution=resolution[1], large_kernel=31, patch_size=16)
        self.cross_atten2 = TransformerFusion(embedding_dim=channels[2], max_resolution=resolution[2], large_kernel=15, patch_size=8)
        self.cross_atten3 = TransformerFusion(embedding_dim=channels[1], max_resolution=resolution[3], large_kernel=7, patch_size=4)
        self.num_classes = num_classes
        self.compute_dtype = torch.bfloat16
        self._cache = PackCache()
        self._cache_f32 = PackCache()

    def _pack(self, dt):
        dev = self.conv4.weight.device
        pc = lambda conv, bn=None, may_pad=False: _PackedConv(conv, bn, dev, may_pad=may_pad, dtype=dt)   # noqa: E731
        p = {"conv4": pc(self.conv4, may_pad=True), "conv3": pc(self.conv3), "conv2": pc(self.conv2), "conv1": pc(self.conv1),
             "conv0": pc(self.conv0)}
        for name in ("up1", "up2", "up3", "up4"):
            net = getattr(self, name)._net
            p[name + "a"] = pc(net[0], net[1], may_pad=True)
            p[name + "b"] = pc(net[3], net[4])
        return p

    def _packed(self, dt):
        if dt == torch.float32:
            return self._cache_f32.get(self, lambda: self._pack(dt))
        return self._cache.get(self, lambda: self._pack(dt))

    def forward_nhwc(self, img_features, hist_features, **kwargs) -> Tuple[torch.Tensor, int, int]:
        """Returns (unet_out [B, H, W, num_classes] channels-last in ``compute_dtype``, H, W)."""
        if self.training:
            raise NotImplementedError("the decoder shell serves eval mode (BatchNorm folded)")
        dt = self.compute_dtype
        if dt not in (torch.bfloat16, torch.float32):
            raise ValueError(f"Decoder.compute_dtype must be torch.bfloat16 or torch.float32, not {dt}")
        f32 = dt == torch.float32
        if f32:
            for name in ("cross_atten1", "cross_atten2", "cross_atten3"):
                if any(p.dtype != torch.float32 for p in getattr(self, name).parameters()):
                    raise ValueError(f"compute_dtype float32 runs the fusion modules' fp32 engine, but {name} has been cast "
                                     "to a lower precision: leave the cross_atten* modules in float32")
        x0, x1, x2, x3, x4 = [t.detach().float().contiguous() for t in img_features]
        f1, f2, f3 = hist_features
        _lib.require_cuda(x4, "img_features")
        dev = x4.device
        B = x4.shape[0]
        P = self._packed(dt)
        L = self.LEAKY
        upcat = "cfp_upsample_concat_f32" if f32 else "cfp_upsample_concat"

        def buf(B, H, W, Cc):
            return torch.empty(B, H, W, Cc, device=dev, dtype=dt)

        with torch.cuda.device(dev):
            st = _lib.stream_ptr

            def to_nhwc(skip, cpad):
                """NCHW fp32 feature -> channels-last, channels zero-padded (cfp_upsample_concat with no low-res map)."""
                Bq, Cq, H, W = skip.shape
                out = buf(Bq, H, W, cpad)
                _lib.call(upcat, 0, 1, 1, 0, 8, skip.data_ptr(), Cq, out.data_ptr(), Bq, H, W, cpad, st())
                return out

            def up(lo, h, w, c_lo, skip, name):
                """UpSampleBN.forward (decoder.py:50-58): resize + concat, conv-BN-LeakyReLU twice."""
                _, Cs, H, W = skip.shape
                pa, pb = P[name + "a"], P[name + "b"]
                cat = buf(B, H, W, pa.cin_pad)
                _lib.call(upcat, lo.data_ptr(), h, w, c_lo, c_lo, skip.data_ptr(), Cs, cat.data_ptr(), B, H, W,
                          pa.cin_pad, st())
                y = buf(B, H, W, pa.cout)
                _conv(pa, cat, B, H, W, L, y, pa.cout, 0)
                z = buf(B, H, W, pb.cout)
                _conv(pb, y, B, H, W, L, z, pb.cout, 0)
                return z, H, W

            def level(z, H, W, pconv, fusion, feat):
                """x_d = conv1x1(z); x_d = cat([x_d, cross_atten(x_d, feat)])  (decoder.py:110-112 and the two below)."""
                Cd = pconv.cout
                cat = buf(B, H, W, 2 * Cd)
                _conv(pconv, z, B, H, W, 1.0, cat, 2 * Cd, 0)
                fusion.forward_tokens(cat, 2 * Cd, B, H, W, feat, cat, 2 * Cd, Cd, **kwargs)
                return cat, 2 * Cd

            h4, w4 = x4.shape[2], x4.shape[3]
            d4 = buf(B, h4, w4, P["conv4"].cout)
            _conv(P["conv4"], to_nhwc(x4, P["conv4"].cin_pad), B, h4, w4, 1.0, d4, P["conv4"].cout, 0)
            z, H, W = up(d4, h4, w4, P["conv4"].cout, x3, "up1")
            d3, c3 = level(z, H, W, P["conv3"], self.cross_atten3, f3)
            z, H2, W2 = up(d3, H, W, c3, x2, "up2")
            d2, c2 = level(z, H2, W2, P["conv2"], self.cross_atten2, f2)
            z, H1, W1 = up(d2, H2, W2, c2, x1, "up3")
            d1, c1 = level(z, H1, W1, P["conv1"], self.cross_atten1, f1)
            z, H0, W0 = up(d1, H1, W1, c1, x0, "up4")
            out = buf(B, H0, W0, self.num_classes)
            _conv(P["conv0"], z, B, H0, W0, 1.0, out, self.num_classes, 0)
        return out, H0, W0

    def forward(self, img_features, hist_features, **kwargs):
        out, H, W = self.forward_nhwc(img_features, hist_features, **kwargs)
        B = out.shape[0]
        res = torch.empty(B, self.num_classes, H, W, device=out.device, dtype=out.dtype)
        with torch.cuda.device(out.device):
            _lib.call("cfp_tokens_to_nchw", out.data_ptr(), res.data_ptr(), B, self.num_classes, H, W, _lib.dtype_code(out.dtype),
                      _lib.stream_ptr())
        return res.float()


class DepthRegression(nn.Module):
    """decoder.py:9-37 (parameters; norm = 'linear' is what libcfp serves)."""

    def __init__(self, in_channels, dim_out=256, embedding_dim=128, norm="linear"):
        super().__init__()
        if norm != "linear":
            raise NotImplementedError("libcfp serves DepthRegression with norm='linear' (the reference configs)")
        if in_channels != 128 or embedding_dim != 128:
            raise NotImplementedError("libcfp serves the 128-channel head (deltar.py:16)")
        self.norm = norm
        self.conv3x3 = nn.Conv2d(in_channels, embedding_dim, kernel_size=3, stride=1, padding=1)
        self.conv1x1 = nn.Conv2d(embedding_dim, embedding_dim, kernel_size=1, stride=1, padding=0, bias=False)
        self.regressor = nn.Sequential(nn.Linear(embedding_dim, 256), nn.LeakyReLU(), nn.Linear(256, 256), nn.LeakyReLU(),
                                       nn.Linear(256, dim_out))


class DepthHead(nn.Module):
    """The part of ``Deltar`` below the decoder (deltar.py:16-19, 50-61): ``depth_head`` + ``conv_out`` -> (bin_edges
    [B, n_bins + 1], pred [B, 1, H, W][, prob [B, n_bins, H, W]]).  Consumes the decoder's channels-last map: a bf16 map
    runs the tcgen05 head, an fp32 map the exact fp32 one."""

    def __init__(self, n_bins=256, min_val=1e-3, max_val=10.0, norm="linear"):
        super().__init__()
        if n_bins not in (128, 256):
            raise NotImplementedError("libcfp serves n_bins 128 / 256")
        self.num_classes, self.min_val, self.max_val = n_bins, float(min_val), float(max_val)
        self.depth_head = DepthRegression(128, dim_out=n_bins, norm=norm)
        self.conv_out = nn.Sequential(nn.Conv2d(128, n_bins, kernel_size=1, stride=1, padding=0), nn.Softmax(dim=1))
        self._cache = PackCache()
        self._cache_f32 = PackCache()

    def _pack(self, dt=torch.bfloat16):
        dev = self.conv_out[0].weight.device
        dh = self.depth_head
        f = lambda t: host(t).contiguous().to(dev)                    # noqa: E731
        wout = host(self.conv_out[0].weight)[:, :, 0, 0]                  # [n_bins, 128]
        wout = wout.t() if dt == torch.float32 else umma_block(wout)      # fp32 [128][n_bins] | bf16 UMMA block
        return dict(ram=_PackedConv(dh.conv3x3, None, dev, dtype=dt), wc=f(dh.conv1x1.weight[:, :, 0, 0]),
                    w0=f(dh.regressor[0].weight), b0=f(dh.regressor[0].bias), w2=f(dh.regressor[2].weight),
                    b2=f(dh.regressor[2].bias), w4=f(dh.regressor[4].weight), b4=f(dh.regressor[4].bias),
                    wout=wout.contiguous().to(dev), bout=f(self.conv_out[0].bias))

    def forward_nhwc(self, unet_out: torch.Tensor, H: int, W: int, return_prob: bool = False):
        if self.training:
            raise NotImplementedError("the head serves eval mode")
        _lib.require_cuda(unet_out, "unet_out")
        dt = unet_out.dtype
        if dt == torch.float32:
            P = self._cache_f32.get(self, lambda: self._pack(dt))
            bins, expect = "cfp_head_bins_f32", "cfp_head_expect_f32"
        elif dt == torch.bfloat16:
            P = self._cache.get(self, self._pack)
            bins, expect = "cfp_head_bins", "cfp_head_expect"
        else:
            raise ValueError(f"unet_out must be bfloat16 (tensor-core head) or float32 (exact fp32 head), not {dt}")
        B = unet_out.shape[0]
        dev = unet_out.device
        nb = self.num_classes
        ram = torch.empty(B, H, W, 128, device=dev, dtype=dt)
        mean = torch.empty(B, 128, device=dev, dtype=torch.float32)
        edges = torch.empty(B, nb + 1, device=dev, dtype=torch.float32)
        centres = torch.empty(B, nb, device=dev, dtype=torch.float32)
        pred = torch.empty(B, 1, H, W, device=dev, dtype=torch.float32)
        prob = torch.empty(B, nb, H, W, device=dev, dtype=torch.float32) if return_prob else None
        with torch.cuda.device(dev):
            st = _lib.stream_ptr()
            _conv(P["ram"], unet_out, B, H, W, 1.0, ram, 128, 0)
            _lib.call(bins, unet_out.data_ptr(), 128, B, H * W, 128, P["wc"].data_ptr(), P["w0"].data_ptr(), P["b0"].data_ptr(),
                      P["w2"].data_ptr(), P["b2"].data_ptr(), P["w4"].data_ptr(), P["b4"].data_ptr(), P["w0"].shape[0], nb,
                      C.c_float(self.min_val), C.c_float(self.max_val), mean.data_ptr(), edges.data_ptr(), centres.data_ptr(), st)
            _lib.call(expect, ram.data_ptr(), 128, B, H * W, P["wout"].data_ptr(), P["bout"].data_ptr(), centres.data_ptr(),
                      nb, pred.data_ptr(), _lib.ptr(prob), st)
        return (edges, pred, prob) if return_prob else (edges, pred)
