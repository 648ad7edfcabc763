"""CPU tests of the host side: geometry, drop-in contract (state_dict keys), the C-ABI
library's symbol table, and loud failure without a GPU.  No compute calls."""
import ctypes
import os
import re
import subprocess

import numpy as np
import pytest
import torch

import cfpnet_b200
from cfpnet_b200 import _lib, geometry, synth
from cfpnet_b200.config import args
from helpers import FUSION_CASES as _BASE_CASES, FUSION_CASES_Z6, FusionCase, ref_keys

FUSION_CASES = _BASE_CASES + FUSION_CASES_Z6

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    from cfpnet_b200.build import build
    build()
    return _lib.load()


def test_library_exports_every_declared_symbol(lib):
    header = open(os.path.join(ROOT, "include", "cfp.h")).read()
    declared = sorted(set(re.findall(r"\b(cfp_[a-z0-9_]+)\s*\(", header)))
    assert len(declared) >= 11
    raw = ctypes.CDLL(_lib.LIB_PATH)
    for name in declared:
        assert hasattr(raw, name), f"{name} declared in include/cfp.h but not exported"
        assert name in _lib.SIGNATURES, f"{name} has no ctypes signature"
    # ... and the reverse: an entry point removed from the header must not stay exported
    nm = subprocess.run(["nm", "-D", "--defined-only", _lib.LIB_PATH], capture_output=True, text=True, check=True).stdout
    exported = set(re.findall(r"^\S+\s+T\s+(cfp_[a-z0-9_]+)$", nm, re.M))
    assert exported, nm
    assert not exported - set(declared), f"exported but not declared in include/cfp.h: {sorted(exported - set(declared))}"
    assert lib.cfp_version() == _lib.ABI_VERSION
    assert lib.cfp_last_error() is not None


def test_ctypes_structs_match_header_layout():
    assert ctypes.sizeof(_lib.CfpGeom) == 16 * 4
    assert ctypes.sizeof(_lib.CfpLoftrW) == 11 * 8
    assert ctypes.sizeof(_lib.CfpDapmW) == 17 * 8
    assert ctypes.sizeof(_lib.CfpLkpmW) == 11 * 8         # 10 pointers + int32 (+pad)
    assert ctypes.sizeof(_lib.CfpTwinsW) == 22 * 8 + 5 * 8 + 8
    assert ctypes.sizeof(_lib.CfpHistW) == 19 * 8


def test_workspace_bytes_is_pure_host_arithmetic(lib):
    g = _lib.CfpGeom(zone_num=8, p1=3, p2=3, tzh=24, tzw=24, ry1=24, rx1=24)
    small = lib.cfp_workspace_bytes(1, 26, 34, 128, 6, 7, _lib.CFP_F32, ctypes.byref(g))
    big = lib.cfp_workspace_bytes(4, 26, 34, 128, 6, 7, _lib.CFP_F32, ctypes.byref(g))
    half = lib.cfp_workspace_bytes(4, 26, 34, 128, 6, 0, _lib.CFP_BF16, ctypes.byref(g))
    assert 0 < small < big and half < big


def _centred_geom(zn, p, H, W):
    t = zn * p
    y0, x0 = (H - t) // 2, (W - t) // 2
    return _lib.CfpGeom(zone_num=zn, p1=p, p2=p, sy_wo=y0, sx_wo=x0, ey_wo=y0 + t, ex_wo=x0 + t, tzh=t, tzw=t,
                        ry0=y0, ry1=y0 + t, rx0=x0, rx1=x0 + t)


@pytest.mark.parametrize("zn,p", [(8, 3), (6, 4), (4, 6), (1, 24), (12, 2)])
@pytest.mark.parametrize("dtype", [_lib.CFP_F32, _lib.CFP_BF16])
def test_workspace_covers_every_entry_point(lib, zn, p, dtype):
    """One workspace serves all layer calls of a level.  cfp_twins_fwd / cfp_lkpm_fwd get no geometry and lay it out
    for 64 zones: with the reference's 6x6 training layout the size computed from the geometry alone was smaller and
    both calls refused it (the round-1 6x6 failure).  Pure host arithmetic - no device work."""
    B, H, W, C, ws, lk = 2, 26, 34, 128, 6, 7
    g = _centred_geom(zn, p, H, W)
    n = lib.cfp_workspace_bytes(B, H, W, C, ws, lk, dtype, ctypes.byref(g))
    assert n >= lib.cfp_workspace_bytes(B, H, W, C, ws, lk, dtype, None)        # twins / lkpm layouts (subsets of it)
    assert n >= lib.cfp_workspace_bytes(B, H, W, C, ws, 0, dtype, None)
    assert n >= lib.cfp_workspace_bytes(B, H, W, C, 0, lk, dtype, None)
    if zn <= 8:
        assert n == lib.cfp_workspace_bytes(B, H, W, C, ws, lk, dtype, ctypes.byref(_centred_geom(8, 3, H, W)))


@pytest.mark.skipif(torch.cuda.is_available(), reason="calls the layer entry points with fake device pointers: only "
                                                      "safe where the first launch fails (no CUDA driver)")
@pytest.mark.parametrize("zn,p", [(8, 3), (6, 4)])
@pytest.mark.parametrize("dtype", [_lib.CFP_F32, _lib.CFP_BF16])
def test_layer_calls_accept_the_advertised_workspace(lib, zn, p, dtype):
    """Argument validation of the layer calls happens before any CUDA call: with the size cfp_workspace_bytes hands out
    none of them may answer 'workspace too small' (they go on and fail at the first launch - there is no GPU here)."""
    B, H, W, C, ws, lk = 2, 26, 34, 128, 6, 7
    g = _centred_geom(zn, p, H, W)
    n = lib.cfp_workspace_bytes(B, H, W, C, ws, lk, dtype, ctypes.byref(g))
    fake = ctypes.c_void_p(0x1000)
    tw, lkw, dw, lw = _lib.CfpTwinsW(), _lib.CfpLkpmW(), _lib.CfpDapmW(), _lib.CfpLoftrW()
    tw.ws, lkw.ksize = ws, lk
    calls = {
        "twins": lambda: lib.cfp_twins_fwd(fake, B, H, W, C, ctypes.byref(tw), fake, n, dtype, None),
        "lkpm": lambda: lib.cfp_lkpm_fwd(fake, B, H, W, C, ctypes.byref(lkw), fake, n, dtype, None),
        "dapm": lambda: lib.cfp_dapm_fwd(fake, B, H, W, C, ctypes.byref(g), ctypes.byref(dw), fake, n, dtype, None),
        "d2i": lambda: lib.cfp_d2i_fwd(fake, fake, fake, fake, fake, B, H, W, C, 16, ctypes.byref(g), ctypes.byref(lw),
                                       0, fake, n, dtype, None),
    }
    for name, fn in calls.items():
        assert fn() != 0, name                                     # no device: the call cannot succeed ...
        assert b"workspace too small" not in lib.cfp_last_error(), (name, lib.cfp_last_error())   # ... but not for this
    # and one byte less than the geometry-less layout needs is still refused, with the sizes in the message
    assert lib.cfp_lkpm_fwd(fake, B, H, W, C, ctypes.byref(lkw), fake,
                            lib.cfp_workspace_bytes(B, H, W, C, 0, lk, dtype, None) - 1, dtype, None) != 0
    assert b"workspace too small" in lib.cfp_last_error()


def test_rejected_call_sets_thread_local_message(lib):
    rc = lib.cfp_lkpm_fwd(None, 1, 8, 8, 48, None, None, 0, 0, None)
    assert rc != 0 and b"null" in lib.cfp_last_error().lower()
    rc = lib.cfp_lkpm_fwd(ctypes.c_void_p(256), 1, 8, 8, 48, None, None, 0, 0, None)
    assert rc != 0 and b"embedding_dim" in lib.cfp_last_error()
    # a map smaller than the GSA sub-sampling kernel: the reference's strided conv raises, the library refuses
    tw = _lib.CfpTwinsW()
    tw.ws = 6
    rc = lib.cfp_twins_fwd(ctypes.c_void_p(256), 1, 4, 40, 32, ctypes.byref(tw), ctypes.c_void_p(256), 1 << 30, 0, None)
    assert rc != 0 and b"sub-sampling kernel" in lib.cfp_last_error()


@pytest.mark.parametrize("tag", FUSION_CASES)
def test_zone_geometry_matches_reference(tag):
    case = FusionCase(tag)
    inp = case.inputs()
    H, W = synth.level_hw(case.geometry, case.level)
    g = geometry.zone_geometry(inp["patch_info"], case.max_res[1], H, W)
    ref = case.geo
    got = dict(pad_height=g.pad_h, pad_width=g.pad_w, p1=g.p1, p2=g.p2, sy_wo_pad=g.sy_wo, sx_wo_pad=g.sx_wo,
               ey_wo_pad=g.ey_wo, ex_wo_pad=g.ex_wo, sy=g.sy, ey=g.ey, sx=g.sx, ex=g.ex, tzh=g.tzh, tzw=g.tzw,
               interpolate=g.interpolate, zone_num=g.zone_num)
    for k, v in got.items():
        assert v == ref[k], (k, v, ref[k])
    geometry.check_geometry(g, H, W)
    zm = case.mask_bits("zone_mask").reshape(case.batch, H, W)
    rect = np.zeros((H, W), dtype=bool)
    rect[g.ry0:g.ry1, g.rx0:g.rx1] = True
    assert all(np.array_equal(zm[b], rect) for b in range(case.batch))
    assert g.n_inside == int(rect.sum())


def test_patch_info_truncation_and_padding_rules():
    # negative starts truncate toward zero; pads are relative to the hard-coded 480x640 canvas
    rect = synth.centred_rects(480, 640, 64)             # rows -16 .. 496
    pi = geometry.patch_info_from_rect_data(rect)
    assert pi["zone_num"] == 8
    assert pi[16]["pad_size"].tolist() == [1, 0] and pi[4]["pad_size"].tolist() == [4, 0]
    assert pi[16]["index_wo_pad"].tolist() == [-1, 4, 31, 36]
    rect2 = rect.clone()
    rect2[:, 0] += 6                                      # y0 = -10 -> trunc(-10/16) = 0, pad = ceil(10/16) = 1
    rect2[:, 2] += 6
    pi2 = geometry.patch_info_from_rect_data(rect2)
    assert pi2[16]["index_wo_pad"][0].item() == 0 and pi2[16]["pad_size"][0].item() == 2
    assert pi2[16]["patch_size"].tolist() == [4, 4]
    # ragged zones: the largest zone defines the patch size (ceil)
    rect3 = synth.centred_rects(416, 544, 48)
    rect3[5, 2] += 5
    assert geometry.patch_info_from_rect_data(rect3)[16]["patch_size"].tolist() == [4, 3]


def test_check_geometry_rejects_what_the_reference_cannot_run():
    # zones hanging below a 416-row image but inside 480: pad = 0, the canvas slice would be cut short
    rect = synth.centred_rects(416, 544, 48)
    rect[:, 0] += 40
    rect[:, 2] += 40
    pi = geometry.collate_patch_info([geometry.patch_info_from_rect_data(rect)])
    g = geometry.zone_geometry(pi, 40, 26, 34)
    with pytest.raises(ValueError):
        geometry.check_geometry(g, 26, 34)


def test_state_dict_keys_match_reference():
    keys = ref_keys()
    enc = cfpnet_b200.HistogramEncoder()
    assert {k: list(v.shape) for k, v in enc.state_dict().items()} == keys["hist_encoder"]
    saved = list(args.attention_layer)
    try:
        for kind, layers in (("combine1", synth.COMBINE1_LAYERS), ("baseline", synth.BASELINE_LAYERS)):
            args.attention_layer = list(layers)
            for level, (C, _, max_res, lk) in synth.LEVELS.items():
                m = cfpnet_b200.TransformerFusion(C, list(max_res), large_kernel=lk, patch_size=640 // max_res[1])
                mine = {k: list(v.shape) for k, v in m.state_dict().items()}
                assert mine == keys[f"fusion_{kind}_L{level}"], (kind, level)
                m.load_state_dict(synth.synthetic_state_dict(keys[f"fusion_{kind}_L{level}"], seed=level), strict=True)
    finally:
        args.attention_layer = saved


def test_unknown_layer_name_raises_like_reference():
    saved = list(args.attention_layer)
    try:
        args.attention_layer = ["hist2image", "bogus"]
        with pytest.raises(NotImplementedError):
            cfpnet_b200.TransformerFusion(32, [120, 160], large_kernel=31, patch_size=4)
    finally:
        args.attention_layer = saved


def test_product_path_has_no_cpu_fallback():
    m = cfpnet_b200.TransformerFusion(128, [30, 40], large_kernel=7, patch_size=4).eval()
    inp = synth.make_inputs("G416", 1, levels=(3,))
    with pytest.raises(_lib.CfpError, match="no CPU implementation"):
        m(inp["x3"], torch.zeros(1, 64, 16, 128), mask=inp["mask"], patch_info=inp["patch_info"],
          rect_data=inp["rect_data"], rgb=None)
    enc = cfpnet_b200.HistogramEncoder().eval()
    with pytest.raises(_lib.CfpError, match="no CPU implementation"):
        enc(inp["hist_data"].unsqueeze(-1))
    with pytest.raises(_lib.CfpError, match="no CPU implementation"):          # train mode is CUDA-only too
        enc.train()(inp["hist_data"].unsqueeze(-1))


def test_product_package_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "cfpnet_b200")
    for root, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(root, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle|cfp_oracle|import_module\(.oracle", src, re.M), f


def test_synthetic_inputs_are_deterministic():
    a, b = synth.make_inputs("G416", 2, levels=(3,)), synth.make_inputs("G416", 2, levels=(3,))
    assert torch.equal(a["x3"], b["x3"]) and torch.equal(a["hist_data"], b["hist_data"])
    assert torch.equal(a["mask"], b["mask"])
    assert (a["hist_data"][~a["mask"]] == 0).all()
    assert 0.6 < a["mask"].float().mean() < 0.95


def test_fastdiv_multiply_high_formula_is_exact():
    """providers.cuh: FastDiv::div(n) = umul64hi(n, ~0ull / d + 1) for 0 <= n < 2^32 - the kernels' only division.
    Checked against Python integers on the divisors the path uses (window / zone / frame sizes) and random ones."""
    import random
    rng = random.Random(0)
    divisors = [1, 2, 3, 9, 16, 36, 48, 81, 96, 136, 138, 144, 308, 576, 884, 1232, 2304, 3536, 4928, 9216, 14144] + \
               [rng.randrange(1, 1 << 20) for _ in range(200)]
    for d in divisors:
        m = ((1 << 64) - 1) // d + 1 if d > 1 else 0
        ns = [0, 1, d - 1, d, d + 1, 2 * d - 1, (1 << 32) - 1, (1 << 31), (1 << 31) - 1] + [rng.randrange(0, 1 << 32) for _ in range(300)]
        for n in ns:
            n &= (1 << 32) - 1
            q = n if d == 1 else (n * m) >> 64
            assert q == n // d, (n, d)
    # conv3x3_tc's 32-bit magic: umulhi(i, ceil(2^32 / WP)) == i / WP whenever i * WP < 2^32
    for WP in (36, 70, 138, 162, 642):
        magic = ((1 << 32) + WP - 1) // WP
        for i in list(range(0, 5000)) + [rng.randrange(0, (1 << 32) // WP) for _ in range(2000)]:
            assert (i * magic) >> 32 == i // WP, (i, WP)


@pytest.mark.parametrize("tag", FUSION_CASES)
def test_zone_masks_kernel_formula_matches_reference_masks(tag):
    """csrc/k_layout.cu::zone_masks_kernel restated index by index in numpy (zone_mask: rectangle test per cell;
    hist_mask[j] = mask[j // (p1 p2)]; pad_mask: in-image part of the canvas) against the masks the reference
    materialised - the kernel's arithmetic checked without a GPU, for the 8x8 and the 6x6 zone layouts."""
    case = FusionCase(tag)
    inp = case.inputs()
    H, W = synth.level_hw(case.geometry, case.level)
    g = geometry.zone_geometry(inp["patch_info"], case.max_res[1], H, W)
    B, Z, P = case.batch, g.zone_num ** 2, g.p1 * g.p2
    n = np.arange(B * H * W) % (H * W)
    y, x = n // W, n % W
    zone = (y >= g.ry0) & (y < g.ry1) & (x >= g.rx0) & (x < g.rx1)
    hist = inp["mask"].numpy().reshape(-1).astype(bool)[np.arange(B * Z * P) // P]
    j = np.arange(B * g.tzh * g.tzw)
    cx, cy = j % g.tzw, (j // g.tzw) % g.tzh
    pad = np.ones_like(j, dtype=bool)
    if g.pad_h > 0 or g.pad_w > 0:
        top, left = max(-g.sy_wo, 0), max(-g.sx_wo, 0)
        bot, right = max(g.ey_wo - H, 0), max(g.ex_wo - W, 0)
        pad = ~((cy < top) | (cy >= g.tzh - bot) | (cx < left) | (cx >= g.tzw - right))
    assert np.array_equal(zone.reshape(B, H * W), case.mask_bits("zone_mask"))
    assert np.array_equal(hist.reshape(B * Z, P), case.mask_bits("hist_mask"))
    assert np.array_equal(pad.reshape(B, g.tzh, g.tzw), case.mask_bits("pad_mask"))


def test_header_constants_match_the_host_side():
    from cfpnet_b200 import headers
    src = open(os.path.join(ROOT, "include", "cfp.h")).read()
    for name, val in (("CFP_SUMSQ_FLOATS", headers.SUMSQ_FLOATS), ("CFP_SILOG_SCRATCH_DOUBLES", headers.SILOG_SCRATCH_DOUBLES),
                      ("CFP_METRICS_SCRATCH_DOUBLES", headers.METRICS_SCRATCH_DOUBLES)):
        m = re.search(r"#define\s+%s\s+(\d+)" % name, src)
        assert m and int(m.group(1)) == val, name


def test_cuda_ops_and_the_torch_stand_in_expose_the_same_interface():
    """train_seq.py is written once against an ops interface: the product's CudaOps (libcfp kernels) and the CPU test's
    TorchOps (plain torch, float64) must offer the same methods with the same parameters, or the CPU pin of the
    sequencing would not be a pin of what runs on the GPU."""
    import inspect
    import sys
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from torch_ops import TorchOps
    from cfpnet_b200.train import CudaOps
    pub = lambda cls: {n: f for n, f in inspect.getmembers(cls, inspect.isfunction) if not n.startswith("_")}   # noqa: E731
    a, b = pub(CudaOps), pub(TorchOps)
    assert set(a) == set(b), (sorted(set(a) - set(b)), sorted(set(b) - set(a)))
    for n in a:
        pa, pb = list(inspect.signature(a[n]).parameters), list(inspect.signature(b[n]).parameters)
        assert len(pa) == len(pb), (n, pa, pb)
    used = set(re.findall(r"ops\.([a-z_0-9]+)\(", open(os.path.join(ROOT, "cfpnet_b200", "train_seq.py")).read()))
    assert used <= set(a), sorted(used - set(a))
