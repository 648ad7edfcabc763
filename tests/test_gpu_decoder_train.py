"""The decoder shell and adaptive-bins head in TRAIN mode on the GPU: each new kernel against fp64 (weight gradient, input
gradient through the packed forward conv, upsample adjoint, head backward), then the whole model below the image encoder
(histogram encoder + Decoder with its three fusion calls + DepthHead + SILogLoss, forward and backward) against fp64
autograd of the oracle on the same inputs and positional-encoding draws, the profiler's view of one step, the FlatTrainer
cache invalidation, and the refusals.  Tolerances: rel-L2 <= 1e-4 for the weight gradient (at most 16 x 208 x 272 fp32
products per output), 1e-5 for the input gradient (the forward conv's bound), 1e-3 per tensor for the whole step (the
training bar of DESIGN.md section 8)."""
import pytest
import torch
import torch.nn.functional as F

import cfpnet_b200
from cfpnet_b200 import _lib, decoder as D, decoder_train as DT, synth
from cfpnet_b200.loss import SILogLoss
from cfpnet_b200.train import FlatTrainer
from cfpnet_b200.config import args
from helpers import rel_l2
from oracle import cfp_oracle as O
from test_decoder_train_host import CONV_SHAPES, decoder_shell_train
from test_depth_golden import MAX_VAL, MIN_VAL, tail_state
from test_gpu_decoder_f32 import VENDOR

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
TOL = 1e-3
torch.backends.cudnn.allow_tf32 = False
torch.backends.cuda.matmul.allow_tf32 = False


def _nhwc(t):
    return t.permute(0, 2, 3, 1).contiguous().to(DEV)


WGRAD_CASES = [(ci, co, k, 13, 17, 2) for ci, co, k in CONV_SHAPES] + [
    (80, 32, 3, 208, 272, 1), (32, 32, 3, 208, 272, 2), (128, 128, 3, 208, 272, 1), (128, 256, 1, 208, 272, 2),
    (64, 32, 3, 45, 37, 1), (32, 64, 1, 45, 37, 2)]


@pytest.mark.parametrize("cin,cout,k,H,W,B", WGRAD_CASES)
def test_conv_wgrad_matches_fp64(cin, cout, k, H, W, B):
    g = torch.Generator().manual_seed(cin + 3 * cout + k + H)
    x = torch.randn(B, cin, H, W, generator=g)
    dy = torch.randn(B, cout, H, W, generator=g)
    xd, dyd = _nhwc(x), _nhwc(dy)
    with torch.cuda.device(0):
        a = DT.conv_wgrad(xd, dyd, B, H, W, k)
        b = DT.conv_wgrad(xd, dyd, B, H, W, k)
    torch.cuda.synchronize()
    want = torch.nn.grad.conv2d_weight(x.double(), (cout, cin, k, k), dy.double(), padding=k // 2)
    err = rel_l2(a, want)
    print(f"conv_wgrad_f32 cin {cin} cout {cout} k {k} {H}x{W} B {B}: rel-L2 vs fp64 {err:.2e}")
    assert err <= 1e-4, err
    assert torch.equal(a, b), "two launches differ"


@pytest.mark.parametrize("cin,cout,k", [(80, 32, 3), (168, 64, 3), (232, 256, 1), (312, 128, 3), (392, 256, 3)])
def test_conv_dgrad_through_the_packed_forward_conv(cin, cout, k):
    g = torch.Generator().manual_seed(cin + cout)
    B, H, W = 2, 26, 34
    weight = torch.randn(cout, cin, k, k, generator=g) / (cin * k * k) ** 0.5
    dy = torch.randn(B, cout, H, W, generator=g)
    with torch.cuda.device(0):
        dx = DT.conv_dgrad(_nhwc(dy), weight.to(DEV), B, H, W)
        dx2 = DT.conv_dgrad(_nhwc(dy), weight.to(DEV), B, H, W)
    torch.cuda.synchronize()
    assert dx.shape == (B, H, W, cin) and dx.stride(2) == DT.dgrad_slices(cin)[1]
    want = torch.nn.grad.conv2d_input((B, cin, H, W), weight.double(), dy.double(), padding=k // 2)
    err = rel_l2(dx.permute(0, 3, 1, 2), want)
    print(f"conv dgrad {cin} <- {cout} k {k}: rel-L2 vs fp64 {err:.2e}")
    assert err <= 1e-5, err
    assert torch.equal(dx, dx2)


@pytest.mark.parametrize("h,w,H,W,c_lo,c_skip", [(13, 17, 26, 34, 256, 136), (26, 34, 52, 68, 256, 56), (52, 68, 104, 136, 128, 40),
                                                (104, 136, 208, 272, 64, 16), (13, 17, 13, 17, 0, 232), (15, 20, 30, 40, 256, 136),
                                                (7, 5, 23, 9, 8, 4)])
def test_upsample_concat_adjoint_matches_fp64(h, w, H, W, c_lo, c_skip):
    g = torch.Generator().manual_seed(h + W)
    B = 2
    pitch = c_lo + c_skip + 24                                  # a padded input-gradient buffer
    lo = torch.randn(B, max(c_lo, 4), h, w, generator=g, dtype=torch.float64)[:, :c_lo].requires_grad_(True)
    skip = torch.randn(B, c_skip, H, W, generator=g, dtype=torch.float64, requires_grad=True)
    dcat = torch.randn(B, H, W, pitch, generator=g)
    outs = []
    for _ in range(2):
        d_lo = torch.full((B, h, w, c_lo), float("nan"), device=DEV)
        d_skip = torch.full((B, c_skip, H, W), float("nan"), device=DEV)
        with torch.cuda.device(0):
            _lib.call("cfp_tr_upsample_concat_bwd_f32", dcat.to(DEV).data_ptr(), pitch, d_lo.data_ptr(), h, w, c_lo, d_skip.data_ptr(),
                      c_skip, B, H, W, _lib.stream_ptr())
        torch.cuda.synchronize()
        outs.append((d_lo, d_skip))
    parts = [skip] if c_lo == 0 else [F.interpolate(lo, size=[H, W], mode="bilinear", align_corners=True), skip]
    torch.cat(parts, dim=1).backward(dcat[..., :c_lo + c_skip].double().permute(0, 3, 1, 2))
    if c_lo:
        err = rel_l2(outs[0][0].permute(0, 3, 1, 2), lo.grad)
        print(f"upsample adjoint {h}x{w} -> {H}x{W}: d_lo rel-L2 vs fp64 {err:.2e}")
        assert err <= 1e-5, err
    assert torch.equal(outs[0][1].cpu().double(), skip.grad)
    assert all(torch.equal(a, b) for a, b in zip(outs[0], outs[1])), "two launches differ"


def _head(sd):
    head = D.DepthHead(n_bins=256, min_val=MIN_VAL, max_val=MAX_VAL)
    head.load_state_dict({k: v for k, v in sd.items() if k.startswith(("depth_head.", "conv_out."))}, strict=True)
    return head.to(DEV)


@pytest.mark.parametrize("scale", [0.5, 8.0])          # 8.0: a peaked softmax (pred close to one bin centre)
def test_head_backward_matches_fp64_autograd(scale):
    sd = tail_state()
    head = _head(sd).train()
    g = torch.Generator().manual_seed(9)
    B, H, W = 2, 40, 56
    unet = (torch.randn(B, 128, H, W, generator=g) * scale)
    u = unet.to(DEV).requires_grad_(True)
    ct_e = torch.randn(B, 257, generator=g)
    ct_p = torch.randn(B, 1, H, W, generator=g)
    edges, pred = head(u)
    (edges * ct_e.to(DEV)).sum().add((pred * ct_p.to(DEV)).sum()).backward()
    torch.cuda.synchronize()
    ref = {k: v.double().requires_grad_(True) for k, v in sd.items() if k.startswith(("depth_head.", "conv_out."))}
    u64 = unet.double().requires_grad_(True)
    we, wp = O.depth_tail(ref, u64, MIN_VAL, MAX_VAL)
    ((we * ct_e.double()).sum() + (wp * ct_p.double()).sum()).backward()
    assert rel_l2(edges, we.detach()) <= 1e-5 and rel_l2(pred, wp.detach()) <= 1e-5
    errs = {"d_unet": rel_l2(u.grad, u64.grad)}
    for n, p in head.named_parameters():
        errs[n] = rel_l2(p.grad, ref[n].grad)
    for n, e in errs.items():
        print(f"head backward (scale {scale}) {n}: rel-L2 vs fp64 {e:.2e}")
    assert max(errs.values()) <= 1e-4, errs


# ---------------------------------------------------------------------------------------------- whole model
def _model(sd):
    enc = cfpnet_b200.HistogramEncoder()
    enc.load_state_dict({k[len("hist_encoder."):]: v for k, v in sd.items() if k.startswith("hist_encoder.")}, strict=True)
    dec = D.Decoder(num_classes=128)
    dec.load_state_dict({k[len("decoder."):]: v for k, v in sd.items() if k.startswith("decoder.")}, strict=True)
    return enc.to(DEV).train(), dec.to(DEV).train(), _head(sd).train()


def _target(geometry, B):
    img_h, img_w, _ = synth.GEOMETRIES[geometry]
    return torch.rand(B, 1, img_h, img_w, generator=torch.Generator().manual_seed(31)) * 4 + 0.5


def _cuda_step(enc, dec, head, geometry, B, seed=5):
    inp = synth.make_inputs(geometry, B, seed=seed, levels=())
    feats = [t.to(DEV).requires_grad_(True) for t in synth.encoder_features(geometry, B, seed=seed)]
    hist = enc(inp["hist_data"].to(DEV).unsqueeze(-1))
    torch.manual_seed(2)                                   # positional-encoding crops, drawn in call order L3, L2, L1
    unet = dec(feats, hist, rect_data=inp["rect_data"], mask=inp["mask"].to(DEV), patch_info=inp["patch_info"], rgb=None)
    edges, pred = head(unet)
    loss = SILogLoss()(pred, _target(geometry, B).to(DEV))
    loss.backward()
    return inp, feats, edges, pred, loss


def _oracle_step(sd, geometry, B, inp, dt):
    """fp64 (or fp32) autograd of the oracle on the GPU: hist_encoder -> decoder shell with its three fusion calls ->
    depth_tail -> silog_loss, train-mode BatchNorm; same inputs and positional-encoding draws as ``_cuda_step``."""
    ref = {k: (v.to(DEV) if v.dtype == torch.long else v.to(DEV, dt).requires_grad_("running" not in k)) for k, v in sd.items()}
    feats = [t.to(DEV, dt).requires_grad_(True) for t in synth.encoder_features(geometry, B, seed=5)]
    mask = inp["mask"].to(DEV)
    max_res = {n: mr for n, _, mr, _ in O.LEVELS}
    stats = {}

    def fuse(name, x, feat1):
        return O.transformer_fusion(O.sub(ref, f"decoder.{name}."), synth.COMBINE1_LAYERS, max_res[name], x, feat1, mask,
                                    inp["patch_info"], bn_stats=stats)

    hist = O.hist_encoder(O.sub(ref, "hist_encoder."), inp["hist_data"].to(DEV, dt), bn_stats=stats)
    torch.manual_seed(2)
    unet = decoder_shell_train(O.sub(ref, "decoder."), feats, hist, fuse, stats)
    edges, pred = O.depth_tail(ref, unet, MIN_VAL, MAX_VAL)
    loss = O.silog_loss(pred, _target(geometry, B).to(DEV, dt))
    loss.backward()
    out = {"loss": loss.detach().reshape(1), "pred": pred.detach(), "bin_edges": edges.detach()}
    out.update({f"img_features[{i}]": f.grad for i, f in enumerate(feats)})
    out.update({n: t.grad for n, t in ref.items() if t.is_floating_point() and t.requires_grad})
    return out, stats


@pytest.mark.parametrize("geometry", ["G416", "G416z6"])
def test_whole_model_train_step_matches_fp64_oracle(geometry):
    """Every tensor within rel-L2 1e-3 of fp64, or within 4x of what fp32 autograd of the same oracle (torch, TF32 off)
    deviates from fp64: in train mode the regressor's channel mean sends a per-channel near-constant gradient into the
    up-sampling blocks, which the batch-statistics BatchNorm backward removes again - a cancellation that amplifies any
    fp32 evaluation's rounding (and the fp32 atomics of the existing BatchNorm / bias reductions) to ~1e-3."""
    saved = list(args.attention_layer)
    try:
        args.attention_layer = list(synth.COMBINE1_LAYERS)
        sd = tail_state()
        enc, dec, head = _model(sd)
        B = 2
        inp, feats, edges, pred, loss = _cuda_step(enc, dec, head, geometry, B)
        torch.cuda.synchronize()
        want, stats = _oracle_step(sd, geometry, B, inp, torch.float64)
        f32, _ = _oracle_step(sd, geometry, B, inp, torch.float32)

        got = {"loss": loss.detach().reshape(1), "pred": pred.detach(), "bin_edges": edges.detach()}
        got.update({f"img_features[{i}]": f.grad for i, f in enumerate(feats)})
        params = {}
        for prefix, mod in (("hist_encoder.", enc), ("decoder.", dec), ("", head)):
            params.update({prefix + n: p for n, p in mod.named_parameters()})
        zero_like = []
        for n, p in params.items():
            if want.get(n) is None:
                assert p.grad is None, f"{n}: never reached by the reference, must keep grad None"
                continue
            assert p.grad is not None, f"{n}: received no gradient"
            sib = want.get(n[:-len("bias")] + "weight") if n.endswith(".bias") else None
            if sib is not None and float(want[n].norm()) <= 1e-8 * float(sib.norm()):
                # a conv bias feeding a batch-statistics BatchNorm: zero gradient in exact arithmetic
                zero_like.append(n)
                assert float(p.grad.norm()) <= TOL * float(sib.norm()), (n, float(p.grad.norm()), float(sib.norm()))
                continue
            got[n] = p.grad
        bufs = dict(list(enc.named_buffers(prefix="hist_encoder")) + list(dec.named_buffers(prefix="decoder")))
        errs, bounds = {}, {}
        for n, v in stats.items():
            if v.dtype == torch.int64:
                assert int(bufs[n]) == int(v), n
            else:
                errs["buffer " + n], bounds["buffer " + n] = rel_l2(bufs[n], v), TOL
        for n, t in got.items():
            errs[n] = rel_l2(t, want[n])
            bounds[n] = max(TOL, 4 * rel_l2(f32[n], want[n]))
        worst = max(errs, key=lambda k: errs[k] / bounds[k])
        n_over = sum(1 for k in errs if errs[k] > TOL)
        print(f"{geometry} B {B}: {len(errs)} tensors, {len(zero_like)} zero-gradient biases; loss {float(loss):.6f} vs "
              f"{float(want['loss']):.6f}; pred {errs['pred']:.2e}, bin_edges {errs['bin_edges']:.2e}; worst {worst} {errs[worst]:.2e} "
              f"(fp32 torch {rel_l2(f32[worst], want[worst]):.2e}); {n_over} tensors above 1e-3, median "
              f"{sorted(errs.values())[len(errs) // 2]:.2e}")
        assert any(k.startswith("decoder.up4") for k in errs) and any(k.startswith("depth_head") for k in errs)
        assert len([k for k in errs if k.startswith("buffer decoder.up")]) == 16
        assert errs["loss"] <= 1e-5 and errs["pred"] <= 1e-5 and errs["bin_edges"] <= 1e-5
        bad = {k: (errs[k], bounds[k]) for k in errs if not errs[k] <= bounds[k]}
        assert not bad, bad
    finally:
        args.attention_layer = saved


def test_train_step_runs_no_vendor_kernel():
    saved = list(args.attention_layer)
    try:
        args.attention_layer = list(synth.COMBINE1_LAYERS)
        enc, dec, head = _model(tail_state())
        _cuda_step(enc, dec, head, "G416", 1)
        torch.cuda.synchronize()
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            _cuda_step(enc, dec, head, "G416", 1)
            torch.cuda.synchronize()
        names = {e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA}
        foreign = sorted(n for n in names if "cfp::" not in n and any(v in n.lower() for v in VENDOR))
        assert not foreign, foreign
        for k in ("conv_wgrad_f32_kernel", "upsample_concat_bwd_f32_kernel", "head_expect_bwd_f32_kernel", "head_bins_bwd_f32_kernel",
                  "conv_f32_kernel", "tr_bn_bwd"):
            assert any(k in n for n in names), k
    finally:
        args.attention_layer = saved


def _eval_fp32(enc, dec, head, seed=7):
    enc.eval(), dec.eval(), head.eval()
    dec.compute_dtype = torch.float32
    inp = synth.make_inputs("G416", 1, seed=seed, levels=())
    feats = [t.to(DEV) for t in synth.encoder_features("G416", 1, seed=seed)]
    with torch.no_grad():
        hist = enc(inp["hist_data"].to(DEV).unsqueeze(-1))
        torch.manual_seed(3)
        unet = dec(feats, hist, rect_data=inp["rect_data"], mask=inp["mask"].to(DEV), patch_info=inp["patch_info"], rgb=None)
        edges, pred = head(unet)
    torch.cuda.synchronize()
    enc.train(), dec.train(), head.train()
    return edges, pred


def test_flat_trainer_step_refreshes_the_fp32_eval_engine():
    """After an optimizer step (raw-pointer writes torch's version counters do not see) the fp32 eval engine of Decoder and
    DepthHead must run on the new weights: bit-identical to a fresh model loaded with the updated state_dict."""
    saved = list(args.attention_layer)
    try:
        args.attention_layer = list(synth.COMBINE1_LAYERS)
        sd = tail_state()
        enc, dec, head = _model(sd)
        trainer = FlatTrainer([enc, dec, head], lr=1e-3)
        for step in range(2):
            trainer.zero_grad()
            _cuda_step(enc, dec, head, "G416", 1, seed=5 + step)
            trainer.update()
            edges, pred = _eval_fp32(enc, dec, head)          # the second step updates weights these packed copies came from
        full = {**{"hist_encoder." + k: v for k, v in enc.state_dict().items()},
                **{"decoder." + k: v for k, v in dec.state_dict().items()}, **head.state_dict()}
        fresh = _model({k: v.cpu() for k, v in full.items()})
        want_edges, want_pred = _eval_fp32(*fresh)
        moved = rel_l2(pred, _eval_fp32(*_model(sd))[1])
        err = max(rel_l2(edges, want_edges), rel_l2(pred, want_pred))
        print(f"fp32 eval after two steps: {err:.2e} from a fresh model with the updated weights (the steps moved it {moved:.2e})")
        assert moved > 1e-4, "the steps changed nothing"
        # the fusion layers' fp32 engine is not bit-reproducible run to run (4e-6 measured): stale packed weights would be
        # off by the step itself
        assert err <= 1e-4, err
    finally:
        args.attention_layer = saved


def test_train_mode_refusals():
    saved = list(args.attention_layer)
    try:
        args.attention_layer = list(synth.COMBINE1_LAYERS)
        sd = tail_state()
        enc, dec, head = _model(sd)
        inp = synth.make_inputs("G416", 1, seed=5, levels=())
        feats = [t.to(DEV) for t in synth.encoder_features("G416", 1, seed=5)]
        hist = [torch.zeros(1, 64, 16, c, device=DEV) for c in (32, 64, 128)]
        kw = dict(rect_data=inp["rect_data"], mask=inp["mask"].to(DEV), patch_info=inp["patch_info"], rgb=None)
        with pytest.raises(_lib.CfpError, match="CUDA device"):
            dec([f.cpu() for f in feats], hist, **kw)
        with pytest.raises(_lib.CfpError, match="fp32"):
            head(torch.zeros(1, 128, 8, 8, device=DEV, dtype=torch.bfloat16))
        dec.up2.to(torch.bfloat16)
        with pytest.raises(_lib.CfpError, match="fp32"):
            dec(feats, hist, **kw)
        _, dec, _ = _model(sd)
        inp = synth.make_inputs("G480", 1, seed=5, levels=())       # 480 x 640: L3 takes hist2image's resize branch
        feats = [t.to(DEV) for t in synth.encoder_features("G480", 1, seed=5)]
        with pytest.raises(NotImplementedError):
            dec(feats, hist, rect_data=inp["rect_data"], mask=inp["mask"].to(DEV), patch_info=inp["patch_info"], rgb=None)
    finally:
        args.attention_layer = saved
