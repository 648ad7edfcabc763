"""Exact fp32 engine of the decoder shell (f1) and adaptive-bins head (f2): each kernel against torch in fp64 on the same fp32
inputs, the head against the fp64 oracle, and the all-fp32 CUDA model below the image encoder (histogram encoder, Decoder
with its three fusion calls, DepthHead) against the reference's depth map (G416) and the fp64 oracle (G480, B = 2).
Tolerances: fp32 accumulation over at most 3528 products per output -> rel-L2 <= 1e-5 per conv; final depth abs-rel
<= 1e-4, the fp32 bound of tests/test_gpu_depth.py."""
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


def nhwc(x_nchw):
    return x_nchw.permute(0, 2, 3, 1).contiguous().to(DEV)


@pytest.mark.parametrize("cin,cout,k,H,W,B,bn,coff", [
    (392, 256, 3, 26, 34, 2, True, 0),             # up1 first conv: 13 K-chunks (the last one partial), cout split over two CTAs
    (256, 128, 1, 26, 34, 2, False, 0),            # conv3: 1 x 1 into the first half of a 256-wide buffer
    (168, 64, 3, 52, 68, 1, True, 64),             # up3 first conv, written into a channel slice
    (80, 32, 3, 104, 136, 1, True, 0),             # up4 first conv
    (32, 128, 3, 208, 272, 1, False, 0),           # conv0 at half resolution
    (128, 128, 3, 45, 37, 1, False, 0),            # odd map: partial last row and column tiles
    (64, 32, 1, 52, 68, 2, False, 32),             # conv1: 1 x 1 to 32 channels, into the second half of a buffer
])
def test_conv_f32_matches_fp64(cin, cout, k, H, W, B, bn, coff):
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
    pc = D._PackedConv(conv, norm, DEV, dtype=torch.float32)
    assert pc.cin_pad == cin
    x = torch.randn(B, cin, H, W, generator=g)
    xin = nhwc(x)
    pitch = cout + coff + 8
    outs = []
    for _ in range(2):
        out = torch.full((B, H, W, pitch), 7.0, device=DEV)
        with torch.cuda.device(0):
            D._conv(pc, xin, B, H, W, 0.01, out, pitch, coff)
        torch.cuda.synchronize()
        outs.append(out)
    # fp64 on the same fp32 operands (BatchNorm folded into the fp32 weights as the host packs them)
    w = conv.weight.detach()
    shift = conv.bias.detach()
    if bn:
        scale, sh = D.fold_bn(norm)
        w = w * scale[:, None, None, None]
        shift = sh + conv.bias.detach() * scale
    want = F.conv2d(x.double(), w.double(), None, padding=k // 2) + shift.double()[None, :, None, None]
    want = F.leaky_relu(want, 0.01).permute(0, 2, 3, 1)
    out = outs[0]
    got = out[..., coff:coff + cout].double().cpu()
    err = rel_l2(got, want)
    print(f"conv_f32 cin {cin} cout {cout} k {k}: rel-L2 vs fp64 {err:.2e}")
    assert err <= 1e-5, err
    assert (out[..., :coff] == 7.0).all() and (out[..., coff + cout:] == 7.0).all(), "wrote outside its channel slice"
    assert torch.equal(outs[0], outs[1]), "two launches differ"


def test_upsample_concat_f32_matches_torch():
    g = torch.Generator().manual_seed(3)
    B, h, w, H, W, c_lo, c_skip, c_out = 2, 13, 17, 26, 34, 256, 136, 400
    lo = torch.randn(B, c_lo, h, w, generator=g)
    skip = torch.randn(B, c_skip, H, W, generator=g)
    skip_d = skip.to(DEV)
    out = torch.full((B, H, W, c_out), float("nan"), device=DEV)
    with torch.cuda.device(0):
        _lib.call("cfp_upsample_concat_f32", nhwc(lo).data_ptr(), h, w, c_lo, c_lo, skip_d.data_ptr(), c_skip, out.data_ptr(), B, H, W,
                  c_out, _lib.stream_ptr())
    torch.cuda.synchronize()
    up = F.interpolate(lo.double(), size=[H, W], mode="bilinear", align_corners=True)
    want = torch.cat([up, skip.double()], dim=1).permute(0, 2, 3, 1)
    got = out.double().cpu()
    assert rel_l2(got[..., :c_lo + c_skip], want) <= 1e-6, rel_l2(got[..., :c_lo + c_skip], want)
    assert (got[..., c_lo + c_skip:] == 0).all()


def test_upsample_concat_f32_without_low_resolution_map():
    """Decoder.to_nhwc: NCHW feature -> channels-last, zero channels up to the pitch (lo = NULL, c_lo = 0)."""
    g = torch.Generator().manual_seed(4)
    B, C, H, W, cpad = 2, 230, 13, 17, 240
    skip = torch.randn(B, C, H, W, generator=g)
    skip_d = skip.to(DEV)
    out = torch.full((B, H, W, cpad), float("nan"), device=DEV)
    with torch.cuda.device(0):
        _lib.call("cfp_upsample_concat_f32", 0, 1, 1, 0, 8, skip_d.data_ptr(), C, out.data_ptr(), B, H, W, cpad, _lib.stream_ptr())
    torch.cuda.synchronize()
    got = out.cpu()
    assert torch.equal(got[..., :C], skip.permute(0, 2, 3, 1))
    assert (got[..., C:] == 0).all()


def _head(sd):
    head = D.DepthHead(n_bins=256, min_val=MIN_VAL, max_val=MAX_VAL)
    head.load_state_dict({k: v for k, v in sd.items() if k.startswith(("depth_head.", "conv_out."))}, strict=True)
    return head.to(DEV).eval()


def test_head_f32_matches_oracle():
    sd = tail_state()
    head = _head(sd)
    g = torch.Generator().manual_seed(8)
    B, H, W = 2, 40, 56
    unet = torch.randn(B, 128, H, W, generator=g) * 0.5
    with torch.no_grad():
        edges, pred, prob = head.forward_nhwc(nhwc(unet), H, W, return_prob=True)
        edges2, pred2, prob2 = head.forward_nhwc(nhwc(unet), H, W, return_prob=True)
        torch.cuda.synchronize()
        want_edges, want_pred = O.depth_tail({k: v.double() for k, v in sd.items()}, unet.double(), MIN_VAL, MAX_VAL)
    assert edges.dtype == pred.dtype == prob.dtype == torch.float32
    e_err, p_err = rel_l2(edges.double().cpu(), want_edges), O.abs_rel(pred.cpu(), want_pred)
    print(f"fp32 head vs the fp64 oracle: edges rel-L2 {e_err:.2e}, pred abs-rel {p_err:.2e}")
    assert e_err <= 1e-5
    assert p_err <= 1e-5
    assert torch.allclose(prob.sum(1), torch.ones_like(prob.sum(1)), atol=1e-5)
    cen = 0.5 * (edges[:, :-1] + edges[:, 1:])
    assert rel_l2((prob.double() * cen.double()[:, :, None, None]).sum(1, keepdim=True), pred.double()) <= 1e-6
    assert torch.equal(edges, edges2) and torch.equal(pred, pred2) and torch.equal(prob, prob2), "two runs differ"


def _fp32_model(sd):
    dec = D.Decoder(num_classes=128)
    dec.load_state_dict({k[len("decoder."):]: v for k, v in sd.items() if k.startswith("decoder.")}, strict=True)
    dec = dec.to(DEV).eval()
    dec.compute_dtype = torch.float32
    enc = cfpnet_b200.HistogramEncoder()
    enc.load_state_dict({k[len("hist_encoder."):]: v for k, v in sd.items() if k.startswith("hist_encoder.")}, strict=True)
    enc = enc.to(DEV).eval()
    return enc, dec, _head(sd)


def _run_fp32(sd, geometry, B, seed):
    enc, dec, head = _fp32_model(sd)
    inp = synth.make_inputs(geometry, B, seed=seed, levels=())
    feats = [t.to(DEV) for t in synth.encoder_features(geometry, B, seed=seed)]
    with torch.no_grad():
        hist = enc(inp["hist_data"].to(DEV).unsqueeze(-1))
        assert all(h.dtype == torch.float32 for h in hist)
        torch.manual_seed(2)                 # positional-encoding crops, drawn in call order L3, L2, L1
        unet, H, W = dec.forward_nhwc(feats, hist, rect_data=inp["rect_data"], mask=inp["mask"].to(DEV),
                                      patch_info=inp["patch_info"], rgb=None)
        assert unet.dtype == torch.float32
        edges, pred = head.forward_nhwc(unet, H, W)
    torch.cuda.synchronize()
    return inp, edges, pred


# kernels of a vendor library or of torch's own conv / GEMM / softmax / resize: none may run in the fp32 model
VENDOR = ("cudnn", "cutlass", "cublas", "gemm", "xmma", "convolution", "conv2d", "convolve", "softmax", "upsample", "im2col")


def test_whole_fp32_decoder_and_head_final_depth():
    """The north-star check (final depth within 0.5 % abs-rel of the reference) on the all-CUDA fp32 model below the image
    encoder, held to the 1e-4 fp32 bound."""
    saved = list(args.attention_layer)
    try:
        args.attention_layer = list(synth.COMBINE1_LAYERS)
        sd = tail_state()
        _run_fp32(sd, "G416", 1, 5)                               # packs the weights outside the profiled window
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            _, edges, pred = _run_fp32(sd, "G416", 1, 5)
        names = {e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA}
        foreign = sorted(n for n in names if "cfp::" not in n and any(v in n.lower() for v in VENDOR))
        assert not foreign, foreign
        for k in ("conv_f32_kernel", "upsample_concat_f32_kernel", "channel_mean_f32_kernel", "head_expect_f32_kernel",
                  "posenc_tokens_nhwc_f32_kernel", "copy_channels_f32_kernel"):
            assert any(k in n for n in names), k
        z = np.load(os.path.join(GOLDEN, "depth_G416_B1.npz"))
        gt = torch.from_numpy(z["pred"])
        assert tuple(pred.shape) == tuple(gt.shape)
        err = O.abs_rel(pred.cpu(), gt)
        e_err = rel_l2(edges.cpu(), torch.from_numpy(z["bin_edges"]))
        print(f"all-CUDA fp32 decoder + head, final depth abs-rel: {err:.3e}, bin_edges rel-L2: {e_err:.3e}")
        assert e_err <= 1e-4
        assert err <= 1e-4
    finally:
        args.attention_layer = saved


def test_whole_fp32_decoder_and_head_g480_b2_against_fp64_oracle():
    """480 x 640, two frames: L3 takes hist2image's bilinear-resize branch.  Reference: the oracle's decoder shell, fusion
    and head in fp64 on the GPU, on the same inputs and positional-encoding draws."""
    saved = list(args.attention_layer)
    try:
        args.attention_layer = list(synth.COMBINE1_LAYERS)
        sd = tail_state()
        inp, edges, pred = _run_fp32(sd, "G480", 2, 5)
        sdd = {k: (v.to(DEV) if v.dtype == torch.long else v.to(DEV, torch.float64)) for k, v in sd.items()}
        feats = [t.to(DEV, torch.float64) for t in synth.encoder_features("G480", 2, seed=5)]
        mask = inp["mask"].to(DEV)
        max_res = {n: mr for n, _, mr, _ in O.LEVELS}

        def fuse(name, x, feat1):
            return O.transformer_fusion(O.sub(sdd, f"decoder.{name}."), synth.COMBINE1_LAYERS, max_res[name], x, feat1, mask,
                                        inp["patch_info"])

        with torch.no_grad():
            hist = O.hist_encoder(O.sub(sdd, "hist_encoder."), inp["hist_data"].to(DEV, torch.float64))
            torch.manual_seed(2)
            unet = O.decoder_shell(O.sub(sdd, "decoder."), feats, hist, fuse)
            want_edges, want_pred = O.depth_tail(sdd, unet, MIN_VAL, MAX_VAL)
        assert pred.shape == want_pred.shape == (2, 1, 240, 320)
        errs = [O.abs_rel(pred[b].cpu(), want_pred[b].cpu()) for b in range(2)]
        print(f"all-CUDA fp32 model at 480x640, B = 2, final depth abs-rel per frame vs fp64 oracle: "
              f"{errs[0]:.3e}, {errs[1]:.3e}; bin_edges rel-L2 {rel_l2(edges.double().cpu(), want_edges.cpu()):.3e}")
        assert max(errs) <= 1e-4
    finally:
        args.attention_layer = saved


def test_engine_selection():
    dec = D.Decoder(num_classes=128)
    assert dec.compute_dtype == torch.bfloat16
    dec = dec.to(DEV).eval()
    dec.cross_atten2.to(torch.bfloat16)
    dec.compute_dtype = torch.float32
    inp = synth.make_inputs("G416", 1, seed=5, levels=())
    feats = [t.to(DEV) for t in synth.encoder_features("G416", 1, seed=5)]
    hist = [torch.zeros(1, 64, 16, c, device=DEV) for c in (32, 64, 128)]
    with torch.no_grad(), pytest.raises(ValueError, match="cross_atten2"):
        dec.forward_nhwc(feats, hist, rect_data=inp["rect_data"], mask=inp["mask"].to(DEV), patch_info=inp["patch_info"], rgb=None)

    fusion = dec.cross_atten3
    x = torch.zeros(1, 26, 34, 256, device=DEV)
    with torch.no_grad(), pytest.raises(ValueError, match="both bf16 or both fp32"):
        fusion.forward_tokens(x, 256, 1, 26, 34, hist[2], x.bfloat16(), 256, 128, rect_data=inp["rect_data"],
                              mask=inp["mask"].to(DEV), patch_info=inp["patch_info"], rgb=None)
