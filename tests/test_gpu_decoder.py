"""Decoder shell (f1) and adaptive-bins head (f2) kernels: each op against plain torch fp32 ops on the same bf16-rounded
operands (the torch fp32 reference of a floating-point kernel), the bin regressor / fused softmax-expectation head against
the oracle's restatement of DepthRegression + conv_out (pinned on the reference by tests/test_depth_golden.py), and the
whole CUDA decoder + head against the reference's own depth map (tests/golden/depth_G416_B1.npz).
Tolerances: one bf16 rounding of the output (2^-9) on top of fp32 accumulation -> rel-L2 <= 5e-3 per op."""
import os

import numpy as np
import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

import cfpnet_b200
from cfpnet_b200 import _lib, decoder as D, synth
from cfpnet_b200.config import args
from helpers import rel_l2
from oracle import cfp_oracle as O
from test_depth_golden import GOLDEN, MAX_VAL, MIN_VAL, tail_state

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
torch.backends.cudnn.allow_tf32 = False
torch.backends.cuda.matmul.allow_tf32 = False


def nhwc_bf16(x_nchw, cpad):
    B, C, H, W = x_nchw.shape
    out = torch.zeros(B, H, W, cpad, device=DEV, dtype=torch.bfloat16)
    out[..., :C] = x_nchw.permute(0, 2, 3, 1).to(DEV, torch.bfloat16)
    return out


@pytest.mark.parametrize("cin,cout,k,H,W,B,bn,may_pad,coff", [
    (392, 256, 3, 26, 34, 2, True, True, 0),       # up1 first conv: 5 K-chunks of 80, N = 256 (512 TMEM columns)
    (256, 128, 1, 26, 34, 2, False, False, 0),     # conv3: 1 x 1 into the first half of a 256-wide buffer
    (168, 64, 3, 52, 68, 1, True, True, 64),       # up3 first conv: padded to 192, four M-tiles, two column slices
    (80, 32, 3, 104, 136, 1, True, True, 0),       # up4 first conv: three column slices of 46
    (32, 128, 3, 208, 272, 1, False, False, 0),    # conv0 at half resolution: eight column slices, rows not a tile multiple
    (128, 128, 3, 45, 37, 1, False, False, 0),     # odd map: partial last row tile and partial last column slice
])
def test_conv_fwd_matches_torch(cin, cout, k, H, W, B, bn, may_pad, coff):
    g = torch.Generator().manual_seed(cin + cout + k)
    conv = nn.Conv2d(cin, cout, k, padding=k // 2)
    with torch.no_grad():
        conv.weight.copy_(torch.randn(conv.weight.shape, generator=g) / (cin * k * k) ** 0.5)
        conv.bias.copy_(torch.randn(cout, generator=g) * 0.3)
    norm = None
    if bn:
        norm = nn.BatchNorm2d(cout).eval()
        with torch.no_grad():
            norm.weight.copy_(torch.rand(cout, generator=g) + 0.5)
            norm.bias.copy_(torch.randn(cout, generator=g) * 0.2)
            norm.running_mean.copy_(torch.randn(cout, generator=g) * 0.2)
            norm.running_var.copy_(torch.rand(cout, generator=g) + 0.5)
    pc = D._PackedConv(conv, norm, DEV, may_pad=may_pad)
    x = torch.randn(B, cin, H, W, generator=g)
    xin = nhwc_bf16(x, pc.cin_pad)
    pitch = cout + coff + 8
    out = torch.full((B, H, W, pitch), 7.0, device=DEV, dtype=torch.bfloat16)
    with torch.cuda.device(0):
        D._conv(pc, xin, B, H, W, 0.01, out, pitch, coff)
    torch.cuda.synchronize()
    # torch fp32 on the same bf16-rounded operands (BatchNorm folded into the weights as the host packs them)
    w = conv.weight.detach()
    shift = conv.bias.detach()
    if bn:
        scale, sh = D.fold_bn(norm)
        w = w * scale[:, None, None, None]
        shift = sh + conv.bias.detach() * scale
    want = F.conv2d(x.bfloat16().float(), w.bfloat16().float(), None, padding=k // 2) + shift[None, :, None, None]
    want = F.leaky_relu(want, 0.01).permute(0, 2, 3, 1)
    got = out[..., coff:coff + cout].float().cpu()
    assert rel_l2(got, want) <= 5e-3, rel_l2(got, want)
    assert (out[..., :coff] == 7.0).all() and (out[..., coff + cout:] == 7.0).all(), "wrote outside its channel slice"


def test_bf16_upsample_concat_matches_torch():
    g = torch.Generator().manual_seed(3)
    B, h, w, H, W, c_lo, c_skip, c_out = 2, 13, 17, 26, 34, 256, 136, 400
    lo = torch.randn(B, c_lo, h, w, generator=g)
    skip = torch.randn(B, c_skip, H, W, generator=g)
    lo_t = nhwc_bf16(lo, c_lo)
    out = torch.empty(B, H, W, c_out, device=DEV, dtype=torch.bfloat16)
    with torch.cuda.device(0):
        _lib.call("cfp_upsample_concat", lo_t.data_ptr(), h, w, c_lo, c_lo, skip.to(DEV).data_ptr(), c_skip, out.data_ptr(), B, H, W,
                  c_out, _lib.CFP_BF16, _lib.stream_ptr())
    torch.cuda.synchronize()
    up = F.interpolate(lo.bfloat16().float(), size=[H, W], mode="bilinear", align_corners=True)
    want = torch.cat([up, skip], dim=1).permute(0, 2, 3, 1)
    got = out.float().cpu()
    assert rel_l2(got[..., :c_lo + c_skip], want) <= 4e-3
    assert (got[..., c_lo + c_skip:] == 0).all()


def _head(sd):
    head = D.DepthHead(n_bins=256, min_val=MIN_VAL, max_val=MAX_VAL)
    head.load_state_dict({k: v for k, v in sd.items() if k.startswith(("depth_head.", "conv_out."))}, strict=True)
    return head.to(DEV).eval()


def test_head_matches_oracle():
    sd = tail_state()
    head = _head(sd)
    g = torch.Generator().manual_seed(8)
    B, H, W = 2, 40, 56
    unet = (torch.randn(B, 128, H, W, generator=g) * 0.5).bfloat16().float()
    with torch.no_grad():
        edges, pred, prob = head.forward_nhwc(nhwc_bf16(unet, 128), H, W, return_prob=True)
        torch.cuda.synchronize()
        want_edges, want_pred = O.depth_tail({k: v.double() for k, v in sd.items()}, unet.double(), MIN_VAL, MAX_VAL)
    assert rel_l2(edges.cpu(), want_edges) <= 1e-4            # mean over bf16 inputs, fp32 regressor
    assert torch.allclose(prob.sum(1), torch.ones_like(prob.sum(1)), atol=1e-4)
    cen = 0.5 * (edges[:, :-1] + edges[:, 1:])
    assert rel_l2((prob * cen[:, :, None, None]).sum(1, keepdim=True), pred) <= 1e-5
    err = O.abs_rel(pred.cpu(), want_pred)
    print(f"head abs-rel vs the fp64 oracle (bf16 range-attention maps): {err:.3e}")
    assert err <= 3e-2


def test_whole_decoder_and_head_final_depth():
    """hist encoder -> Decoder (f1 + the three fusion calls) -> DepthHead (f2), every op a libcfp kernel, against the
    reference's own depth map.  bf16 end to end: at random init the softmax head amplifies feature error ~3x (see
    tests/test_gpu_depth.py); stated tolerance for the all-bf16 model: 2.5 x the deviation of the reference with only its
    fusion modules cast to bf16."""
    saved = list(args.attention_layer)
    try:
        args.attention_layer = list(synth.COMBINE1_LAYERS)
        sd = tail_state()
        dec = D.Decoder(num_classes=128)
        dec.load_state_dict({k[len("decoder."):]: v for k, v in sd.items() if k.startswith("decoder.")}, strict=True)
        dec = dec.to(DEV).eval()
        for m in (dec.cross_atten1, dec.cross_atten2, dec.cross_atten3):
            m.to(torch.bfloat16)
        head = _head(sd)
        enc = cfpnet_b200.HistogramEncoder()
        enc.load_state_dict({k[len("hist_encoder."):]: v for k, v in sd.items() if k.startswith("hist_encoder.")}, strict=True)
        enc = enc.to(DEV).eval()
        enc.out_dtype = torch.bfloat16
        inp = synth.make_inputs("G416", 1, seed=5, levels=())
        feats = [t.to(DEV) for t in synth.encoder_features("G416", 1, seed=5)]
        with torch.no_grad():
            hist = enc(inp["hist_data"].to(DEV).unsqueeze(-1))
            torch.manual_seed(2)
            unet, H, W = dec.forward_nhwc(feats, hist, rect_data=inp["rect_data"], mask=inp["mask"].to(DEV),
                                          patch_info=inp["patch_info"], rgb=None)
            edges, pred = head.forward_nhwc(unet, H, W)
        torch.cuda.synchronize()
        z = np.load(os.path.join(GOLDEN, "depth_G416_B1.npz"))
        gt = torch.from_numpy(z["pred"])
        assert tuple(pred.shape) == tuple(gt.shape)
        err = O.abs_rel(pred.cpu(), gt)
        print(f"all-CUDA bf16 decoder + head, final depth abs-rel: {err:.3e} (reference with bf16 fusion modules: {float(z['ref_bf16_abs_rel']):.3e})")
        assert rel_l2(edges.cpu(), torch.from_numpy(z["bin_edges"])) <= 2e-2
        assert err <= 2.5 * float(z["ref_bf16_abs_rel"])
    finally:
        args.attention_layer = saved
