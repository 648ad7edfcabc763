"""Per-layer checks through the C ABI: each bf16 (tensor-core) layer entry point against the
fp32 (exact FFMA) entry point of the same library on identical inputs, and against the oracle."""
import ctypes

import pytest
import torch

import cfpnet_b200
from cfpnet_b200 import _lib, geometry, synth
from cfpnet_b200.config import args
from helpers import ref_keys, rel_l2
from oracle import cfp_oracle as O

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def module_for(level):
    C, _, max_res, lk = synth.LEVELS[level]
    args.attention_layer = list(synth.COMBINE1_LAYERS)
    m = cfpnet_b200.TransformerFusion(C, list(max_res), large_kernel=lk, patch_size=640 // max_res[1])
    sd = synth.synthetic_state_dict(ref_keys()[f"fusion_combine1_L{level}"], seed=level)
    m.load_state_dict(sd)
    return m.to(DEV).eval(), sd


def layer_call(m, name, layer_idx, feat0, geom_name="G416", level=3, mask=None, feat1=None, poison=False):
    """Run ONE layer entry point in place on a copy of feat0 [B,N,C]; returns the result."""
    C = m.embedding_dim
    H, W = synth.level_hw(geom_name, level)
    B = feat0.shape[0]
    inp = synth.make_inputs(geom_name, B, levels=())
    g = geometry.zone_geometry(inp["patch_info"], m.max_resolution[1], H, W)
    cg = _lib.CfpGeom.from_geometry(g)
    code = _lib.dtype_code(feat0.dtype)
    packed, pos, pos2, _keep = m._cache.get(m, m._pack)
    lib = _lib.load()
    nbytes = lib.cfp_workspace_bytes(B, H, W, C, m.ws, m.large_kernel, code, ctypes.byref(cg))
    work = torch.empty(nbytes, device=DEV, dtype=torch.uint8)
    if poison:
        work.fill_(0xFF)
    x = feat0.clone()
    st = _lib.stream_ptr()
    w = packed[layer_idx]
    if name == "dapm":
        _lib.call("cfp_dapm_fwd", x.data_ptr(), B, H, W, C, ctypes.byref(cg), ctypes.byref(w[0]), work.data_ptr(),
                  nbytes, code, st)
    elif name == "lkpm":
        _lib.call("cfp_lkpm_fwd", x.data_ptr(), B, H, W, C, ctypes.byref(w[1]), work.data_ptr(), nbytes, code, st)
    elif name == "twins":
        _lib.call("cfp_twins_fwd", x.data_ptr(), B, H, W, C, ctypes.byref(w), work.data_ptr(), nbytes, code, st)
    elif name == "d2i":
        _lib.call("cfp_d2i_fwd", x.data_ptr(), x.data_ptr(), feat1.data_ptr(), pos2, mask.data_ptr(),
                  B, H, W, C, feat1.shape[2], ctypes.byref(cg), ctypes.byref(w), 0, work.data_ptr(), nbytes, code, st)
    torch.cuda.synchronize()
    return x, g


@pytest.fixture(autouse=True)
def _restore_flags():
    saved = (list(args.attention_layer), args.change_embedding, args.no_skip_inside)
    yield
    args.attention_layer, args.change_embedding, args.no_skip_inside = saved


@pytest.mark.parametrize("level", [3, 2, 1])
@pytest.mark.parametrize("name,idx", [("dapm", 1), ("lkpm", 1), ("twins", 2), ("d2i", 0)])
def test_bf16_layer_matches_fp32_layer(level, name, idx):
    m, sd = module_for(level)
    C = m.embedding_dim
    H, W = synth.level_hw("G416", level)
    B = 2
    g0 = torch.Generator().manual_seed(level * 10 + idx)
    f32 = torch.randn(B, H * W, C, generator=g0).to(DEV)
    bf = f32.to(torch.bfloat16)
    kw = {}
    if name == "d2i":
        inp = synth.make_inputs("G416", B, levels=())
        kw["mask"] = inp["mask"].to(DEV, torch.uint8).contiguous()
        feat1 = torch.randn(B, 64, 16, C, generator=g0).to(DEV)
        kw["feat1"] = feat1
    exact, geom = layer_call(m, name, idx, bf.float(), level=level, **kw)
    if name == "d2i":
        kw["feat1"] = kw["feat1"].to(torch.bfloat16)
    fast, _ = layer_call(m.to(torch.bfloat16), name, idx, bf, level=level, **kw)
    err = rel_l2(fast, exact)
    assert err <= 1.5e-2, f"{name} L{level}: bf16 vs fp32 rel-L2 {err:.3e}"


@pytest.mark.parametrize("geom,level,B", [("G480", 1, 1), ("G480", 2, 3), ("G480", 3, 2), ("G416", 2, 5), ("G416", 1, 2)])
def test_lkpm_bf16_other_shapes(geom, level, B):
    """LKPM on the tensor-core depthwise path at the shapes the golden cases do not reach: a map that fills the
    120-row M block exactly (480x640 at 1/4), two frames stacked in one plane with an odd batch, row pitches that are
    not a multiple of 8; the workspace is pre-filled with NaN bit patterns (stale bytes must not enter an MMA)."""
    m, sd = module_for(level)
    C = m.embedding_dim
    H, W = synth.level_hw(geom, level)
    f32 = torch.randn(B, H * W, C, generator=torch.Generator().manual_seed(7 * level + B)).to(DEV)
    bf = f32.to(torch.bfloat16)
    exact, _ = layer_call(m, "lkpm", 1, bf.float(), geom_name=geom, level=level)
    fast, _ = layer_call(m.to(torch.bfloat16), "lkpm", 1, bf, geom_name=geom, level=level, poison=True)
    err = rel_l2(fast, exact)
    assert torch.isfinite(fast.float()).all()
    assert err <= 1.5e-2, f"lkpm {geom} L{level} B={B}: bf16 vs fp32 rel-L2 {err:.3e}"


@pytest.mark.parametrize("level", [3, 2, 1])
def test_dapm_layer_vs_oracle(level):
    m, sd = module_for(level)
    C = m.embedding_dim
    H, W = synth.level_hw("G416", level)
    f = torch.randn(2, H * W, C, generator=torch.Generator().manual_seed(level)).to(DEV)
    out, g = layer_call(m, "dapm", 1, f, level=level)
    truth = O.dapm(O.sub(sd, "layers.1.transformer_path."), f.double().cpu(), g.asdict(), H, W)
    assert rel_l2(out, truth) <= 1e-4


@pytest.mark.parametrize("level,dtype", [(3, torch.bfloat16), (2, torch.bfloat16), (1, torch.bfloat16), (3, torch.float32)])
def test_last_layer_nchw_epilogue_equals_layer_then_transpose(level, dtype):
    """cfp_twins_nchw_fwd (the GSA chain's last epilogue stores the caller's NCHW map) against cfp_twins_fwd followed by
    cfp_tokens_to_nchw on the same input: the same arithmetic, only the store differs.  The LSA state of the bf16 engine is
    accumulated with fp32 atomics (windows straddle tiles), so two runs agree to rounding, not bit for bit: 2e-3 rel-L2
    (bf16 output resolution 4e-3); the fp32 engine is deterministic here."""
    m, _ = module_for(level)
    m = m.to(dtype)
    C = m.embedding_dim
    H, W = synth.level_hw("G416", level)
    B = 3
    feat0 = (torch.randn(B, H * W, C, generator=torch.Generator().manual_seed(5)) * 0.5).to(dtype).to(DEV)
    two_step, _ = layer_call(m, "twins", 2, feat0, level=level)
    code = _lib.dtype_code(dtype)
    want = torch.empty(B, C, H, W, device=DEV, dtype=dtype)
    _lib.call("cfp_tokens_to_nchw", two_step.data_ptr(), want.data_ptr(), B, C, H, W, code, _lib.stream_ptr())
    packed, _pos, _pos2, _keep = m._cache.get(m, m._pack)
    lib = _lib.load()
    nbytes = lib.cfp_workspace_bytes(B, H, W, C, m.ws, m.large_kernel, code, None)
    work = torch.empty(nbytes, device=DEV, dtype=torch.uint8)
    x = feat0.clone()
    got = torch.full((B, C, H, W), float("nan"), device=DEV, dtype=dtype)
    _lib.call("cfp_twins_nchw_fwd", x.data_ptr(), got.data_ptr(), B, H, W, C, ctypes.byref(packed[2]), work.data_ptr(), nbytes, code,
              _lib.stream_ptr())
    torch.cuda.synchronize()
    assert torch.isfinite(got.float()).all()
    assert rel_l2(got.float(), want.float()) <= (2e-3 if dtype == torch.bfloat16 else 1e-6)
    with pytest.raises(_lib.CfpError):                      # the result map must not alias the token map
        _lib.call("cfp_twins_nchw_fwd", x.data_ptr(), x.data_ptr(), B, H, W, C, ctypes.byref(packed[2]), work.data_ptr(), nbytes, code,
                  _lib.stream_ptr())

