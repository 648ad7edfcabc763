"""Host side of the whole-model CUDA graph (no GPU needed): argument checks of the NHWC positional-encoding entry point with
device-resident crop offsets, and the capture guard of cfpnet_b200.pipeline.make_graphed_depth on CPU modules."""
import pytest
import torch

import cfpnet_b200
from cfpnet_b200 import _lib, decoder as D, synth
from cfpnet_b200.config import args
from cfpnet_b200.pipeline import _CaptureGuard

FAKE = 256                      # a non-null "device pointer": every call below is refused before anything is launched


@pytest.mark.parametrize("dtype", [_lib.CFP_BF16, _lib.CFP_F32], ids=["bf16", "f32"])
def test_crop_entry_points_refuse_bad_arguments(dtype):
    ok = dict(x=FAKE, pitch=128, pos=FAKE, tok=FAKE, B=1, C=64, H=26, W=34, ph=30, pw=40, oy=0, ox=0, crop=FAKE, dtype=dtype)

    def call(**kw):
        a = {**ok, **kw}
        _lib.call("cfp_posenc_tokens_nhwc_fwd", a["x"], a["pitch"], a["pos"], a["tok"], a["B"], a["C"], a["H"], a["W"], a["ph"],
                  a["pw"], a["oy"], a["ox"], a["crop"], a["dtype"], 0)

    for bad, match in ((dict(x=0), "null pointer"), (dict(pos=0), "null pointer"), (dict(tok=0), "null pointer"),
                       (dict(B=0), "bad shape"), (dict(H=31), "larger than"), (dict(W=41), "larger than"),
                       (dict(oy=1), "host crop offsets"), (dict(ox=2), "host crop offsets"),
                       (dict(crop=0, ox=7), "outside the 30x40 table"), (dict(dtype=2), "unsupported dtype 2"),
                       (dict(C=6), "C = 6"), (dict(pitch=130), "pitch 130"), (dict(C=256), "C = 256")):
        with pytest.raises(_lib.CfpError, match=match):
            call(**bad)


@pytest.fixture()
def model():
    saved = list(args.attention_layer)
    args.attention_layer = list(synth.COMBINE1_LAYERS)
    try:
        yield cfpnet_b200.HistogramEncoder().eval(), D.Decoder(num_classes=128).eval(), D.DepthHead().eval()
    finally:
        args.attention_layer = saved


def _refused(model, change, match):
    enc, dec, head = model
    guard = _CaptureGuard(model, dec, enc)
    guard.check()
    change(enc, dec, head)
    with pytest.raises(_lib.CfpError, match=match):
        guard.check()


def test_guard_refuses_an_in_place_weight_change(model):
    def change(enc, dec, head):
        with torch.no_grad():
            dec.conv0.bias.add_(1)
    _refused(model, change, "changed since capture")


def test_guard_refuses_replaced_tensors_and_submodules(model):
    _refused(model, lambda e, d, h: setattr(d.cross_atten1, "positional_encodings",
                                            torch.nn.Parameter(d.cross_atten1.positional_encodings.detach().clone())),
             "replaced since capture")
    _refused(model, lambda e, d, h: setattr(h, "conv_out", torch.nn.Sequential(torch.nn.Conv2d(128, 256, 1), torch.nn.Softmax(1))),
             "replaced since capture")


def test_guard_refuses_train_mode_and_engine_changes(model):
    _refused(model, lambda e, d, h: d.cross_atten3.layers.train(), "training mode")
    model[1].eval()
    _refused(model, lambda e, d, h: setattr(d, "compute_dtype", torch.float32), "engine or configuration changed")
    _refused(model, lambda e, d, h: setattr(e, "out_dtype", torch.bfloat16), "engine or configuration changed")


def test_guard_refuses_invalidated_packs(model):
    enc, dec, head = model
    dec._cache.get(dec, lambda: "packed")                # stands in for the packed copy a warm-up leaves behind
    guard = _CaptureGuard(model, dec, enc)
    assert ["packed"] == [v for c, _ in guard.caches for _, v in c.held()]
    guard.check()
    dec._cache.invalidate()
    with pytest.raises(_lib.CfpError, match="invalidated or re-packed"):
        guard.check()


def test_guard_refuses_changed_global_flags(model):
    for flag in ("no_skip_inside", "change_embedding"):
        saved = getattr(args, flag)
        try:
            _refused(model, lambda e, d, h: setattr(args, flag, not saved), "engine or configuration changed")
        finally:
            setattr(args, flag, saved)


def test_guard_catches_slot_writes_without_a_registration(model):
    """nn.Module._apply (.to(), .half()) writes the parameter / buffer dicts directly, without a registration hook."""
    bn = model[1].up1._net[1]
    _refused(model, lambda e, d, h: bn._buffers.__setitem__("running_mean", bn.running_mean.clone()), "replaced since capture")
    conv = model[2].conv_out[0]
    _refused(model, lambda e, d, h: conv._parameters.__setitem__("weight", torch.nn.Parameter(conv.weight.detach().clone())),
             "replaced since capture")


def test_guard_fast_path_survives_unrelated_registrations(model):
    enc, dec, head = model
    guard = _CaptureGuard(model, dec, enc)
    torch.nn.Linear(4, 4)                                # registers parameters on a module the graph does not use
    guard.check()
    dec.conv0 = torch.nn.Conv2d(32, 128, 3, padding=1)   # ... and a replaced submodule after that is still caught
    with pytest.raises(_lib.CfpError, match="replaced since capture"):
        guard.check()


def test_guard_holds_the_scratch_tensors(model):
    enc, dec, head = model
    work = torch.empty(16)
    dec.cross_atten2._scratch.get(0, ("key",), lambda t: True, lambda: (work, torch.empty(4)))
    guard = _CaptureGuard(model, dec, enc)
    assert any(t is work for entries in guard.held for _, tensors in entries
               if isinstance(tensors, tuple) for t in tensors)
