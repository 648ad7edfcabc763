"""The model below the image encoder as one CUDA graph (cfpnet_b200.pipeline.make_graphed_depth): the NHWC positional-encoding
entry with device-resident crop offsets against the same entry with host offsets, graph replay against the eager sequence
(histogram encoder -> Decoder.forward_nhwc -> DepthHead.forward_nhwc) on both engines, positional-encoding draws per replay,
ownership of the memory the graph reads, and the staleness checks that refuse a replay."""
import gc

import pytest
import torch

import cfpnet_b200
from cfpnet_b200 import _lib, decoder as D, synth
from cfpnet_b200.config import args
from cfpnet_b200.pipeline import make_graphed_depth
from helpers import rel_l2
from oracle import cfp_oracle as O
from test_depth_golden import MAX_VAL, MIN_VAL, tail_state

pytestmark = pytest.mark.gpu
DEV = "cuda:0"

# Neither engine is bit-reproducible from run to run: the fusion modules reduce their attention state with fp32 atomics on both
# engines (csrc/k_loftr.cu, csrc/k_chain_tc.cu), so replay and eager are compared by tolerance, and each test records the spread
# between two eager runs beside it.  Measured on an NVIDIA B200 (1000 W power limit), two eager runs of the same forward:
# - fp32: pred within 6.5e-6 abs-rel and bin edges within 2.7e-7 rel-L2, held to the project's fp32 bound on final depth
#   (tests/test_gpu_depth.py); the peaked 256-bin probability volume differed by up to 7.9e-4 rel-L2, held to 5x that.
# - bf16: the softmax head amplifies the last-bit differences through bf16 activations: up to 4.0e-2 pred abs-rel, so the
#   pred bound is twice that spread (the bin edges stayed within 2e-5 rel-L2).
FP32_TOL = 1e-4
FP32_PROB_REL_L2 = 4e-3
BF16_PRED_ABS_REL = 8e-2
BF16_EDGES_REL_L2 = 5e-3


def diffs(got, want):
    """(bin_edges rel-L2, pred abs-rel[, prob rel-L2])."""
    d = [rel_l2(got[0].double().cpu(), want[0].double().cpu()), O.abs_rel(got[1].cpu(), want[1].cpu())]
    if len(got) > 2:
        d.append(rel_l2(got[2].double().cpu(), want[2].double().cpu()))
    return d


def assert_fp32_close(got, want, what):
    d = diffs(got, want)
    print(f"{what}: " + ", ".join(f"{n} {v:.2e}" for n, v in zip(("bin_edges rel-L2", "pred abs-rel", "prob rel-L2"), d)))
    assert max(d[:2]) <= FP32_TOL and (len(d) < 3 or d[2] <= FP32_PROB_REL_L2), (what, d)


@pytest.fixture(scope="module", autouse=True)
def combine1_layers():
    saved = list(args.attention_layer)
    args.attention_layer = list(synth.COMBINE1_LAYERS)
    yield
    args.attention_layer = saved


@pytest.fixture(scope="module")
def sd():
    return tail_state()


def make_model(sd, dtype):
    """(hist_encoder, decoder, head) on cuda:0 in eval mode, set up for the fp32 or the bf16 engine."""
    dec = D.Decoder(num_classes=128)
    dec.load_state_dict({k[len("decoder."):]: v for k, v in sd.items() if k.startswith("decoder.")}, strict=True)
    dec = dec.to(DEV).eval()
    dec.compute_dtype = dtype
    if dtype == torch.bfloat16:
        for m in (dec.cross_atten1, dec.cross_atten2, dec.cross_atten3):
            m.to(torch.bfloat16)
    enc = cfpnet_b200.HistogramEncoder()
    enc.load_state_dict({k[len("hist_encoder."):]: v for k, v in sd.items() if k.startswith("hist_encoder.")}, strict=True)
    enc = enc.to(DEV).eval()
    enc.out_dtype = dtype
    head = D.DepthHead(n_bins=256, min_val=MIN_VAL, max_val=MAX_VAL)
    head.load_state_dict({k: v for k, v in sd.items() if k.startswith(("depth_head.", "conv_out."))}, strict=True)
    return enc, dec, head.to(DEV).eval()


@pytest.fixture(scope="module")
def fp32_model(sd):
    return make_model(sd, torch.float32)


def make_inputs(geometry, B, seed):
    """(img_features, hist_data, mask, patch_info) on cuda:0."""
    inp = synth.make_inputs(geometry, B, seed=seed, levels=())
    feats = [t.to(DEV) for t in synth.encoder_features(geometry, B, seed=seed)]
    return feats, inp["hist_data"].to(DEV), inp["mask"].to(DEV), inp["patch_info"]


def eager(model, feats, hist, mask, patch_info, return_prob=False):
    enc, dec, head = model
    with torch.no_grad():
        h = enc(hist.unsqueeze(-1))
        unet, H, W = dec.forward_nhwc(feats, h, rect_data=None, mask=mask, patch_info=patch_info, rgb=None)
        out = head.forward_nhwc(unet, H, W, return_prob=return_prob)
    torch.cuda.synchronize()
    return [t.clone() for t in out]


def capture(model, inputs, **kw):
    feats, hist, mask, patch_info = inputs
    return make_graphed_depth(*model, feats, hist, mask, patch_info, **kw)


def replay(run, inputs, seed):
    torch.manual_seed(seed)
    out = run(*inputs[:3])
    torch.cuda.synchronize()
    return [t.clone() for t in out]


# ------------------------------------------------------------------------------------------------ kernels
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32], ids=["bf16", "f32"])
def test_device_crop_equals_host_offsets(dtype):
    """x_pitch > C: x is the first C channels of a wider channels-last buffer, as the decoder's concat buffer is."""
    g = torch.Generator().manual_seed(1)
    B, C, pitch, H, W, pos_h, pos_w = 2, 64, 128, 52, 68, 60, 80
    x = torch.randn(B, H, W, pitch, generator=g).to(DEV, dtype)
    pos = torch.randn(pos_h * pos_w, C, generator=g).to(DEV)
    code = _lib.dtype_code(dtype)
    for oy, ox in ((0, 0), (3, 5), (7, 1), (pos_h - H, pos_w - W)):
        want = torch.full((B, H * W, C), float("nan"), device=DEV, dtype=dtype)
        got = torch.full((B, H * W, C), float("nan"), device=DEV, dtype=dtype)
        crop = torch.tensor([oy, ox], dtype=torch.int32, device=DEV)
        with torch.cuda.device(0):
            st = _lib.stream_ptr()
            _lib.call("cfp_posenc_tokens_nhwc_fwd", x.data_ptr(), pitch, pos.data_ptr(), want.data_ptr(), B, C, H, W, pos_h, pos_w,
                      oy, ox, None, code, st)
            _lib.call("cfp_posenc_tokens_nhwc_fwd", x.data_ptr(), pitch, pos.data_ptr(), got.data_ptr(), B, C, H, W, pos_h, pos_w,
                      0, 0, crop.data_ptr(), code, st)
        torch.cuda.synchronize()
        assert torch.equal(got, want), (oy, ox)
        ref = x[..., :C].float() + pos.view(pos_h, pos_w, C)[oy:oy + H, ox:ox + W]
        assert torch.equal(got.float(), ref.to(dtype).float().reshape(B, H * W, C)), (oy, ox)


# ------------------------------------------------------------------------------------------------ replay against eager
@pytest.mark.parametrize("geometry,B,return_prob", [("G480", 1, True), ("G416", 1, False), ("G416", 2, True)])
def test_fp32_replay_matches_eager(fp32_model, geometry, B, return_prob):
    """Replayed on inputs other than the captured ones."""
    run = capture(fp32_model, make_inputs(geometry, B, seed=21), return_prob=return_prob)
    other = make_inputs(geometry, B, seed=22)
    torch.manual_seed(5)
    want = eager(fp32_model, *other, return_prob=return_prob)
    torch.manual_seed(5)
    again = eager(fp32_model, *other, return_prob=return_prob)
    got = replay(run, other, seed=5)
    assert len(got) == (3 if return_prob else 2)
    for g, w in zip(got, want):
        assert g.shape == w.shape and g.dtype == w.dtype == torch.float32
    assert_fp32_close(again, want, f"fp32 {geometry} B={B}, two eager runs")
    assert_fp32_close(got, want, f"fp32 {geometry} B={B}, replay vs eager")


@pytest.mark.parametrize("geometry", ["G480", "G416"])
def test_bf16_replay_matches_eager(sd, geometry):
    model = make_model(sd, torch.bfloat16)
    inputs = make_inputs(geometry, 1, seed=23)
    run = capture(model, inputs)
    torch.manual_seed(5)
    want = eager(model, *inputs)
    torch.manual_seed(5)
    spread = diffs(eager(model, *inputs), want)
    err = diffs(replay(run, inputs, seed=5), want)
    print(f"bf16 {geometry} B=1: replay vs eager bin_edges rel-L2 {err[0]:.2e}, pred abs-rel {err[1]:.2e}; "
          f"two eager runs {spread[0]:.2e}, {spread[1]:.2e}")
    assert err[0] <= BF16_EDGES_REL_L2 and err[1] <= BF16_PRED_ABS_REL


# ------------------------------------------------------------------------------------------------ crops
def test_g416_crops_are_drawn_per_replay(fp32_model):
    inputs = make_inputs("G416", 1, seed=24)
    run = capture(fp32_model, inputs)
    a, a2, b = replay(run, inputs, seed=3), replay(run, inputs, seed=3), replay(run, inputs, seed=4)
    assert_fp32_close(a2, a, "fp32 G416, two replays, same seed")
    moved = diffs(b, a)
    print(f"fp32 G416, replays with seeds 3 and 4: bin_edges rel-L2 {moved[0]:.2e}, pred abs-rel {moved[1]:.2e}")
    assert moved[1] > 100 * FP32_TOL, "different seeds gave the same depth: the crop was frozen into the graph"
    torch.manual_seed(4)
    assert_fp32_close(b, eager(fp32_model, *inputs), "fp32 G416 seed 4, replay vs eager")


@pytest.mark.parametrize("geometry,draws", [("G416", 6), ("G480", 0)])
def test_replay_advances_the_generator_as_eager_does(fp32_model, monkeypatch, geometry, draws):
    inputs = make_inputs(geometry, 1, seed=25)
    run = capture(fp32_model, inputs)
    calls = []
    randint = torch.randint
    monkeypatch.setattr(torch, "randint", lambda *a, **k: calls.append(a) or randint(*a, **k))
    torch.manual_seed(11)
    eager(fp32_model, *inputs)
    want, n_eager = torch.get_rng_state(), len(calls)
    calls.clear()
    replay(run, inputs, seed=11)
    assert len(calls) == n_eager == draws
    assert torch.equal(torch.get_rng_state(), want)


# ------------------------------------------------------------------------------------------------ ownership and staleness
def _scratch_ptrs(model):
    """data_ptr of every fusion module's current scratch tensors (workspace and token map); keeps no reference to them."""
    dec = model[1]
    return {t.data_ptr() for m in (dec.cross_atten1, dec.cross_atten2, dec.cross_atten3) for _, ts in m._scratch.held() for t in ts}


def _live_blocks():
    """Addresses of the caching allocator's blocks that are allocated to a tensor right now."""
    return {b["address"] for seg in torch.cuda.memory_snapshot() for b in seg["blocks"] if b["state"] == "active_allocated"}


def test_graph_owns_the_scratch_an_eager_call_evicts(fp32_model):
    """An eager call at another batch size makes every fusion module drop its scratch; the graph reads those tensors, so they
    must stay allocated for as long as `run` exists, and be released with it."""
    inputs = make_inputs("G416", 1, seed=26)
    torch.manual_seed(8)
    want = eager(fp32_model, *inputs)
    run = capture(fp32_model, inputs)
    captured = _scratch_ptrs(fp32_model)
    assert len(captured) == 6
    eager(fp32_model, *make_inputs("G416", 2, seed=27))
    assert not captured & _scratch_ptrs(fp32_model), "the B = 2 forward did not replace the modules' scratch"
    assert captured <= _live_blocks(), "the eviction freed scratch the graph reads"
    got = replay(run, inputs, seed=8)
    assert_fp32_close(got, want, "fp32 G416 B=1 replay after an eager B=2 forward vs eager B=1")
    del run
    gc.collect()
    assert not captured & _live_blocks(), "with the graph gone, the evicted scratch should be released"


def test_stale_replays_are_refused(sd):
    model = make_model(sd, torch.float32)
    enc, dec, head = model
    inputs = make_inputs("G416", 1, seed=28)

    def fresh():
        run = capture(model, inputs)
        replay(run, inputs, seed=1)                                   # a fresh capture replays
        return run

    run = fresh()
    with torch.no_grad():
        dec.conv0.bias.add_(1)
    with pytest.raises(_lib.CfpError, match="changed since capture"):
        run(*inputs[:3])
    run = fresh()                                                     # recapture on the new weights: equals eager on them
    torch.manual_seed(2)
    want = eager(model, *inputs)
    assert_fp32_close(replay(run, inputs, seed=2), want, "fp32 G416, fresh capture on changed weights vs eager")

    dec.cross_atten2._cache.invalidate()                              # what FlatTrainer.update does after an optimizer step
    with pytest.raises(_lib.CfpError, match="invalidated or re-packed"):
        run(*inputs[:3])

    run = fresh()
    head.train()
    with pytest.raises(_lib.CfpError, match="training mode"):
        run(*inputs[:3])
    head.eval()
    replay(run, inputs, seed=1)

    dec.compute_dtype = torch.bfloat16
    with pytest.raises(_lib.CfpError, match="engine or configuration changed"):
        run(*inputs[:3])
    dec.compute_dtype = torch.float32
