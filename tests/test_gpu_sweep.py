"""The fusion layer kernels swept over map shapes and zone layouts the golden cases never reach, against the fp64 oracle,
with per-region error bounds (helpers.region_errors).

Every call goes through the C ABI entry point itself on a workspace filled with 0xFF bytes (NaN bit patterns: a stale
workspace byte that reaches a result shows up).  Both engines run on every case.  The references are the oracle's
per-layer functions in float64; for the bf16 engine they take the bf16 input and the state dict of the bf16-cast module,
upcast - exactly the values the packer receives - so what remains is the kernel's own rounding.

Bounds: fp32 engine rel-L2 <= 2e-5 (measured <= 1e-6 on the whole module).  bf16 engine: the error over the tokens the
layer changes (the bulk) <= BF16_TOL[layer, level]; every region of at least 16 tokens <= 3x the bulk error of the same
call; every token (||out_t - ref_t|| over the frame's RMS token norm) <= 10x the bulk error."""
import ctypes
import functools

import pytest
import torch
import torch.nn.functional as F

import cfpnet_b200
from cfpnet_b200 import _lib, geometry, synth
from cfpnet_b200.config import args
from helpers import check_regions, ref_keys, region_errors
from oracle import cfp_oracle as O
from test_geometry_golden import CASES, grid_rects

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
DTYPES = {"fp32": torch.float32, "bf16": torch.bfloat16}
PREFIX = {"d2i": "layers.0.", "dapm": "layers.1.transformer_path.", "lkpm": "layers.1.large_kernel_path.", "twins": "layers.2."}
FP32_TOL = 2e-5
# bf16 engine, bulk rel-L2 per (layer, level): min(1e-2, 3x the largest value measured over this file's sweep).  Measured
# maxima (NVIDIA B200, 1000 W power limit), bulk rel-L2 / largest region over bulk / largest token over bulk:
#   lkpm   L1 2.94e-3 / 1.05 / 2.3   L2 3.34e-3 / 1.04 / 1.9   L3 3.11e-3 / 1.02 / 1.4
#   twins  L1 4.78e-3 / 1.29 / 3.0   L2 4.29e-3 / 1.27 / 1.8   L3 4.00e-3 / 1.13 / 1.5
#   d2i    L1 3.44e-3 / 1.74 / 5.0   L2 3.35e-3 / 1.58 / 2.8   L3 3.39e-3 / 1.38 / 2.8
#   dapm   L1 3.12e-3 / 1.02 / 2.0   L2 3.10e-3 / 1.03 / 1.8   L3 3.13e-3 / 1.03 / 1.5
#   fusion L1 6.98e-3 / 1.09 / 2.4   L2 6.84e-3 / 1.04 / 1.9   L3 6.95e-3 / 1.02 / 1.5
# fp32 engine on the same cases: bulk rel-L2 <= 3.4e-6 (d2i L1), <= 1.6e-6 on the whole module.
BF16_TOL = {
    ("lkpm", 1): 8.8e-3, ("lkpm", 2): 1e-2, ("lkpm", 3): 9.3e-3,
    ("twins", 1): 1e-2, ("twins", 2): 1e-2, ("twins", 3): 1e-2,
    ("d2i", 1): 1e-2, ("d2i", 2): 1e-2, ("d2i", 3): 1e-2,
    ("dapm", 1): 9.4e-3, ("dapm", 2): 9.3e-3, ("dapm", 3): 9.4e-3,
    ("fusion", 1): 1e-2, ("fusion", 2): 1e-2, ("fusion", 3): 1e-2,
}


@pytest.fixture(autouse=True)
def _restore_flags():
    saved = (list(args.attention_layer), args.change_embedding, args.no_skip_inside)
    yield
    args.attention_layer, args.change_embedding, args.no_skip_inside = saved


@functools.lru_cache(maxsize=None)
def module(level, engine):
    """(TransformerFusion of the level in the engine's dtype, its state dict as float64 CPU tensors)."""
    C, _, max_res, lk = synth.LEVELS[level]
    saved = list(args.attention_layer)
    args.attention_layer = list(synth.COMBINE1_LAYERS)
    m = cfpnet_b200.TransformerFusion(C, list(max_res), large_kernel=lk, patch_size=640 // max_res[1])
    args.attention_layer = saved
    m.load_state_dict(synth.synthetic_state_dict(ref_keys()[f"fusion_combine1_L{level}"], seed=level))
    m = m.to(DEV).to(DTYPES[engine]).eval()
    return m, {k: v.detach().cpu().double() for k, v in m.state_dict().items()}


def layer_call(m, name, x, H, W, cg=None, emb=None, feat1=None, mask=None, assign=0, out_nchw=None):
    """One layer entry point on a copy of ``x`` [B, H*W, C] (B, H, W and the zone geometry ``cg`` chosen by the caller);
    the workspace is refilled with 0xFF on every call."""
    B, C = x.shape[0], m.embedding_dim
    code = _lib.dtype_code(x.dtype)
    packed, _pos, pos2, _keep = m._cache.get(m, m._pack)
    lib = _lib.load()
    nbytes = lib.cfp_workspace_bytes(B, H, W, C, m.ws, m.large_kernel, code, ctypes.byref(cg) if cg is not None else None)
    work = torch.full((nbytes,), 0xFF, device=DEV, dtype=torch.uint8)
    y = x.clone()
    st = _lib.stream_ptr()
    if name == "lkpm":
        _lib.call("cfp_lkpm_fwd", y.data_ptr(), B, H, W, C, ctypes.byref(packed[1][1]), work.data_ptr(), nbytes, code, st)
    elif name == "twins" and out_nchw is not None:
        _lib.call("cfp_twins_nchw_fwd", y.data_ptr(), out_nchw.data_ptr(), B, H, W, C, ctypes.byref(packed[2]), work.data_ptr(),
                  nbytes, code, st)
    elif name == "twins":
        _lib.call("cfp_twins_fwd", y.data_ptr(), B, H, W, C, ctypes.byref(packed[2]), work.data_ptr(), nbytes, code, st)
    elif name == "dapm":
        _lib.call("cfp_dapm_fwd", y.data_ptr(), B, H, W, C, ctypes.byref(cg), ctypes.byref(packed[1][0]), work.data_ptr(), nbytes,
                  code, st)
    elif name == "d2i":
        e = y if emb is None else emb
        _lib.call("cfp_d2i_fwd", y.data_ptr(), e.data_ptr(), feat1.data_ptr(), pos2, mask.data_ptr(), B, H, W, C, feat1.shape[2],
                  ctypes.byref(cg), ctypes.byref(packed[0]), assign, work.data_ptr(), nbytes, code, st)
    torch.cuda.synchronize()
    return y


def judge(out, ref, B, H, W, regions, layer, level, engine, what, bulk=None):
    """fp32: bulk rel-L2 <= FP32_TOL.  bf16: bulk rel-L2 <= BF16_TOL, regions <= 3x bulk, tokens <= 10x bulk."""
    C = ref.shape[-1]
    assert torch.isfinite(out.float()).all(), what
    rep = region_errors(out.reshape(B, H, W, C), ref.reshape(B, H, W, C), regions, bulk)
    print(f"measured {layer} L{level} {engine} bulk {rep['bulk']:.3e} region/bulk {rep['ratio']:.2f} "
          f"token/bulk {rep['token'] / max(rep['bulk'], 1e-30):.2f}  {what}")
    if engine == "fp32":
        assert rep["bulk"] <= FP32_TOL, f"{what}: rel-L2 {rep['bulk']:.3e}"
        return
    assert rep["bulk"] <= BF16_TOL[layer, level], f"{what}: rel-L2 {rep['bulk']:.3e} > {BF16_TOL[layer, level]:.1e}"
    check_regions(rep, what)


def randn(*shape, seed):
    return torch.randn(*shape, generator=torch.Generator().manual_seed(seed))


# ------------------------------------------------------------------ regions
def mask_of(B, H, W, b=None, rows=slice(None), cols=slice(None)):
    m = torch.zeros(B, H, W, dtype=torch.bool)
    m[slice(None) if b is None else b, rows, cols] = True
    return m


def frame_regions(B, H, W):
    return {f"frame {b}": mask_of(B, H, W, b) for b in range(B)}


def tile_regions(B, H, W):
    """Raster 128-token tiles over the whole batch (an M tile of the token-major GEMMs; one may straddle frames)."""
    flat = torch.arange(B * H * W).reshape(B, H, W) // 128
    return {f"tile {t}": flat == t for t in range(int(flat.max()) + 1)}


def lkpm_regions(B, H, W, k):
    """Frames, tiles, the four halo bands of width (k - 1) / 2 of every frame (the first and last rows of a frame stacked
    in a plane, and the zero columns of the plane), the last 32-column tile of the Toeplitz GEMM."""
    p = (k - 1) // 2
    regs = {**frame_regions(B, H, W), **tile_regions(B, H, W)}
    for b in range(B):
        regs[f"frame {b} top band"] = mask_of(B, H, W, b, rows=slice(0, p))
        regs[f"frame {b} bottom band"] = mask_of(B, H, W, b, rows=slice(max(H - p, 0), H))
        regs[f"frame {b} left band"] = mask_of(B, H, W, b, cols=slice(0, p))
        regs[f"frame {b} right band"] = mask_of(B, H, W, b, cols=slice(max(W - p, 0), W))
        regs[f"frame {b} last 32-column strip"] = mask_of(B, H, W, b, cols=slice((W - 1) // 32 * 32, W))
    return regs


def twins_regions(B, H, W, ws):
    """Frames, every LSA window, the windows that hold zero-padding cells, the rows / columns the stride-ws GSA
    sub-sampling conv drops."""
    regs = frame_regions(B, H, W)
    nh, nw = -(-H // ws), -(-W // ws)
    for b in range(B):
        padded = torch.zeros(B, H, W, dtype=torch.bool)
        for i in range(nh):
            for j in range(nw):
                m = mask_of(B, H, W, b, rows=slice(i * ws, (i + 1) * ws), cols=slice(j * ws, (j + 1) * ws))
                regs[f"frame {b} window ({i},{j})"] = m
                if (i + 1) * ws > H or (j + 1) * ws > W:
                    padded |= m
        regs[f"frame {b} windows with padding"] = padded
        regs[f"frame {b} rows the sr conv drops"] = mask_of(B, H, W, b, rows=slice(H // ws * ws, H))
        regs[f"frame {b} columns the sr conv drops"] = mask_of(B, H, W, b, cols=slice(W // ws * ws, W))
    return regs


# ------------------------------------------------------------------ LKPM shapes
LKPM_SHAPES = [
    (1, 1, 120, 160), (1, 2, 104, 136), (1, 3, 52, 68), (1, 4, 30, 40), (1, 5, 15, 20), (1, 1, 7, 9), (1, 2, 33, 150),
    (1, 1, 1, 1),
    (2, 2, 52, 68), (2, 3, 26, 34), (2, 6, 13, 17), (2, 1, 60, 80), (2, 2, 45, 37),
    (3, 2, 26, 34), (3, 1, 30, 40), (3, 3, 13, 17), (3, 2, 12, 16), (3, 1, 33, 41),
]


@pytest.mark.parametrize("engine", ["fp32", "bf16"])
@pytest.mark.parametrize("level,B,H,W", LKPM_SHAPES)
def test_lkpm_sweep(level, B, H, W, engine):
    """L1 (k = 31): the 120-row M block exactly, 2 - 4 frames stacked in a plane (odd B, a partial last stack), a map
    smaller than the padding, W % 32 = 22, one cell.  L2 (k = 15): 3 and 6 stacked frames, odd sizes.  L3 (k = 7): the
    whole-frame tiles, the 16x16 tiles (H * W <= 256), a map over the frame-tile limit."""
    m, sd = module(level, engine)
    C = m.embedding_dim
    x = randn(B, H * W, C, seed=1000 * level + 10 * B + H).to(DTYPES[engine]).to(DEV)
    out = layer_call(m, "lkpm", x, H, W)
    ref = O.lkpm(O.sub(sd, PREFIX["lkpm"]), x.double().cpu(), H, W)
    judge(out, ref, B, H, W, lkpm_regions(B, H, W, m.large_kernel), "lkpm", level, engine, f"lkpm L{level} {engine} B={B} {H}x{W}")


def test_lkpm_too_tall_map_is_refused_before_any_launch():
    """k = 31 on the tensor-core path serves maps up to 120 rows per plane; a taller one is refused up front, and the
    refusal leaves the map and the workspace as they were."""
    m, _ = module(1, "bf16")
    B, H, W, C = 1, 160, 40, 32
    packed, *_ = m._cache.get(m, m._pack)
    lib = _lib.load()
    nbytes = lib.cfp_workspace_bytes(B, H, W, C, m.ws, m.large_kernel, _lib.CFP_BF16, None)
    work = torch.full((nbytes,), 0x5A, device=DEV, dtype=torch.uint8)
    x = randn(B, H * W, C, seed=3).to(torch.bfloat16).to(DEV)
    y = x.clone()
    with pytest.raises(_lib.CfpError, match="too tall"):
        _lib.call("cfp_lkpm_fwd", y.data_ptr(), B, H, W, C, ctypes.byref(packed[1][1]), work.data_ptr(), nbytes, _lib.CFP_BF16,
                  _lib.stream_ptr())
    torch.cuda.synchronize()
    assert torch.equal(y, x) and bool((work == 0x5A).all())


# ------------------------------------------------------------------ Twins shapes
def twins_shapes():
    out = []
    for level, small in ((1, (12, 12)), (2, (9, 13)), (3, (7, 10))):
        ws = O.twins_window_size(synth.LEVELS[level][2])
        th, tw = synth.LEVELS[level][2]
        out += [(level, 3, ws, ws), (level, 2, ws + 1, 2 * ws - 1), (level, 2, 2 * ws, 3 * ws), (level, 1, th, tw),
                (level, 5, *small)]
    return out


@pytest.mark.parametrize("engine", ["fp32", "bf16"])
@pytest.mark.parametrize("level,B,H,W", twins_shapes())
def test_twins_sweep(level, B, H, W, engine):
    """One window, windows with padding on both sides, a whole number of windows, the positional-table size, and a map
    of fewer than 128 tokens (at ws = 12 the least map is 144) at B = 5 so that the 128-row tiles straddle frames.  The
    NCHW-epilogue variant equals the token variant followed by cfp_tokens_to_nchw."""
    m, sd = module(level, engine)
    C, dt = m.embedding_dim, DTYPES[engine]
    x = randn(B, H * W, C, seed=2000 * level + 10 * B + H).mul(0.5).to(dt).to(DEV)
    out = layer_call(m, "twins", x, H, W)
    ref = O.twins_layer(O.sub(sd, PREFIX["twins"]), x.double().cpu(), H, W, m.ws)
    judge(out, ref, B, H, W, twins_regions(B, H, W, m.ws), "twins", level, engine, f"twins L{level} {engine} B={B} {H}x{W}")
    code = _lib.dtype_code(dt)
    want = torch.empty(B, C, H, W, device=DEV, dtype=dt)
    _lib.call("cfp_tokens_to_nchw", out.data_ptr(), want.data_ptr(), B, C, H, W, code, _lib.stream_ptr())
    got = torch.full((B, C, H, W), float("nan"), device=DEV, dtype=dt)
    layer_call(m, "twins", x, H, W, out_nchw=got)
    # the LSA state of the bf16 engine is accumulated with fp32 atomics: two runs agree to rounding (bf16 resolution 4e-3)
    assert torch.isfinite(got.float()).all()
    err = float((got.double() - want.double()).norm() / want.double().norm())
    assert err <= (2e-3 if engine == "bf16" else 1e-6), f"NCHW epilogue vs token layer + transpose: {err:.3e}"


def test_twins_map_smaller_than_the_window_is_refused():
    m, _ = module(3, "fp32")
    with pytest.raises(_lib.CfpError, match="smaller than"):
        layer_call(m, "twins", randn(1, 5 * 40, 128, seed=1).to(DEV), 5, 40)


# ------------------------------------------------------------------ zone layouts: hist2image and DAPM
def served_layouts():
    """(level, image, rects) of every layout of geometry_cases.json the product serves."""
    out = []
    for i, c in enumerate(CASES):
        if "geo" not in c or "reference_raises" in c:
            continue
        _, stride, max_res, _ = synth.LEVELS[c["level"]]
        H, W = c["img"][0] // stride, c["img"][1] // stride
        rect = grid_rects(c)
        g = geometry.zone_geometry(geometry.collate_patch_info([geometry.patch_info_from_rect_data(rect)]), max_res[1], H, W)
        try:
            geometry.check_geometry(g, H, W)
        except ValueError:
            continue
        out.append(pytest.param(c["level"], tuple(c["img"]), rect, "random", id=f"case{i}-L{c['level']}"))
    return out


SERVED = served_layouts()


def rect_grid(y0, x0, ph, pw, zn=8):
    """[zn*zn, 4] rects of zones ph x pw pixels (not necessarily square)."""
    ys = torch.arange(zn, dtype=torch.float32) * ph + y0
    xs = torch.arange(zn, dtype=torch.float32) * pw + x0
    yy, xx = torch.meshgrid(ys, xs, indexing="ij")
    return torch.stack([yy, xx, yy + ph, xx + pw], dim=-1).reshape(-1, 4)


HAND = []
for _lv in (1, 2, 3):
    HAND += [
        # 384x384 image, 8 x 48 px zones: the rectangle is the whole map (DAPM has no outside query)
        pytest.param(_lv, (384, 384), synth.centred_rects(384, 384, 48), "random", id=f"whole_map-L{_lv}"),
        # 48 x 64 px zones (p1 != p2) on 416x544; 40 x 56 px on 480x640 (p1 != p2, resize branch at L3)
        pytest.param(_lv, (416, 544), rect_grid(16, 16, 48, 64), "random", id=f"wide_zones-L{_lv}"),
        pytest.param(_lv, (480, 640), rect_grid(80, 96, 40, 56), "random", id=f"wide_zones_480-L{_lv}"),
        # one frame with every zone invalid, one with every zone valid
        pytest.param(_lv, (416, 544), synth.centred_rects(416, 544, 48), "extremes", id=f"mask_extremes-L{_lv}"),
    ]


def zone_setup(level, img, rects, masks, B, seed):
    _, stride, max_res, _ = synth.LEVELS[level]
    H, W = img[0] // stride, img[1] // stride
    pi = geometry.collate_patch_info([geometry.patch_info_from_rect_data(rects)] * B)
    g = geometry.zone_geometry(pi, max_res[1], H, W)
    geometry.check_geometry(g, H, W)
    Z = g.zone_num ** 2
    if masks == "extremes":
        mask = torch.stack([torch.zeros(Z, dtype=torch.bool), torch.ones(Z, dtype=torch.bool)])
    else:
        mask = torch.rand(B, Z, generator=torch.Generator().manual_seed(seed)) < 0.8
    return H, W, g, mask


def zone_cells(g, B, H, W):
    """[H, W] long: index of the zone a map cell of the rectangle belongs to (canvas position scaled to the zone grid), -1
    outside the rectangle."""
    top, left = max(-g.sy_wo, 0), max(-g.sx_wo, 0)
    ys = torch.arange(g.ry0, g.ry1) - g.ry0 + top
    xs = torch.arange(g.rx0, g.rx1) - g.rx0 + left
    zi = (ys * g.zone_num // g.tzh)[:, None] * g.zone_num + (xs * g.zone_num // g.tzw)[None, :]
    z = torch.full((H, W), -1, dtype=torch.long)
    z[g.ry0:g.ry1, g.rx0:g.rx1] = zi
    return z


def d2i_regions(g, B, H, W, zc):
    regs = {}
    for b in range(B):
        for zi in range(g.zone_num ** 2):
            m = torch.zeros(B, H, W, dtype=torch.bool)
            m[b] = zc == zi
            regs[f"frame {b} zone {zi}"] = m
        border = torch.zeros(H, W, dtype=torch.bool)
        border[g.ry0:g.ry1, g.rx0:g.rx1] = True
        inner = torch.zeros(H, W, dtype=torch.bool)
        inner[g.ry0 + 1:g.ry1 - 1, g.rx0 + 1:g.rx1 - 1] = True
        m = torch.zeros(B, H, W, dtype=torch.bool)
        m[b] = border & ~inner
        regs[f"frame {b} rectangle border"] = m
    return regs


def dapm_regions(g, B, H, W):
    inside = torch.zeros(1, 1, H, W)
    inside[..., g.ry0:g.ry1, g.rx0:g.rx1] = 1
    grow = lambda t: F.max_pool2d(t, 3, stride=1, padding=1)
    inner_ring = (inside * grow(1 - inside))[0, 0].bool()       # inside cells next to an outside cell
    outer_ring = ((1 - inside) * grow(inside))[0, 0].bool()     # outside cells next to an inside cell
    border = torch.ones(H, W, dtype=torch.bool)
    border[1:-1, 1:-1] = False
    ins = inside[0, 0].bool()
    named = {"inside": ins, "outside": ~ins, "inner ring": inner_ring, "outer ring": outer_ring, "map border": border}
    return {k: v.expand(B, H, W) for k, v in named.items()}


def zone_layers(level, img, rects, masks, engine, seed):
    m, sd = module(level, engine)
    C, dt = m.embedding_dim, DTYPES[engine]
    B = 2
    H, W, g, mask = zone_setup(level, img, rects, masks, B, seed)
    cg = _lib.CfpGeom.from_geometry(g)
    Z, S = g.zone_num ** 2, 16
    x = randn(B, H * W, C, seed=seed).to(dt).to(DEV)
    what = f"L{level} {engine} {img[0]}x{img[1]} p={g.p1}x{g.p2} rect [{g.ry0}:{g.ry1},{g.rx0}:{g.rx1}] of {H}x{W} resize={g.interpolate}"

    # ---- DAPM
    out = layer_call(m, "dapm", x, H, W, cg=cg)
    ref = O.dapm(O.sub(sd, PREFIX["dapm"]), x.double().cpu(), g.asdict(), H, W)
    judge(out, ref, B, H, W, dapm_regions(g, B, H, W), "dapm", level, engine, "dapm " + what)

    # ---- hist2image: emb == feat0 with assign = 0 (the fast instantiation), assign = 1 (--no_skip_inside), a separate emb
    feat1 = randn(B, Z, S, C, seed=seed + 1).to(dt).to(DEV)
    emb = randn(B, H * W, C, seed=seed + 2).to(dt).to(DEV)
    ztok = (feat1.double().cpu() + sd["positional_encodings2"]).reshape(B * Z, S, C)
    mask_d = mask.to(DEV, torch.uint8).contiguous()
    zc = zone_cells(g, B, H, W)
    inside = (zc >= 0).reshape(-1)
    invalid_cells = torch.stack([(~mask[b])[zc.clamp_min(0)] & (zc >= 0) for b in range(B)]).reshape(B, -1)
    p = O.sub(sd, PREFIX["d2i"])
    xd = x.double().cpu()
    for assign, sep in ((0, False), (1, False), (0, True)):
        e = emb if sep else None
        out = layer_call(m, "d2i", x, H, W, cg=cg, emb=e, feat1=feat1, mask=mask_d, assign=assign)
        ref = O.hist2image(p, xd, e.double().cpu() if sep else xd, ztok, mask, g.asdict(), H, W, no_skip_inside=bool(assign))
        tag = f"d2i assign={assign} emb={'separate' if sep else 'feat0'} " + what
        o = out.cpu()
        assert torch.equal(o[:, ~inside], x.cpu()[:, ~inside]), f"{tag}: a token outside the zone rectangle changed"
        if not g.interpolate:
            bad = o[invalid_cells]
            want = torch.zeros_like(bad) if assign else x.cpu()[invalid_cells]
            assert torch.equal(bad, want), f"{tag}: cells of invalid zones are not {'zero' if assign else 'the input'}"
        changed = (ref != xd).any(-1).reshape(B, H, W)
        judge(out, ref, B, H, W, d2i_regions(g, B, H, W, zc), "d2i", level, engine, tag, bulk=changed)


@pytest.mark.parametrize("engine", ["fp32", "bf16"])
@pytest.mark.parametrize("level,img,rects,masks", SERVED)
def test_zone_layers_served(level, img, rects, masks, engine):
    """hist2image and DAPM on every layout of tests/golden/geometry_cases.json the product serves (rectangles on the map's
    edges, zones leaving the image, both branches, patch sizes 3 - 18)."""
    zone_layers(level, img, rects, masks, engine, seed=int(rects.sum()) % 9973 + level)


@pytest.mark.parametrize("engine", ["fp32", "bf16"])
@pytest.mark.parametrize("level,img,rects,masks", HAND)
def test_zone_layers_hand(level, img, rects, masks, engine):
    """The rectangle equal to the whole map, non-square zones, a frame with every zone invalid next to one with every
    zone valid."""
    zone_layers(level, img, rects, masks, engine, seed=17 * level + len(masks))


def test_every_served_layout_is_swept():
    assert len(SERVED) == 187


# ------------------------------------------------------------------ the whole TransformerFusion at other image sizes
SIZES = {
    "G384": (384, 384, 48),    # the zone rectangle is the whole map at every level
    "G240": (240, 320, 28),    # 3 frames per plane at L2, the resize branch at L2 and L3
    "G192": (192, 256, 22),    # 16x16 stencil tiles at L3, 4 frames per plane at L2, 2 at k = 31, resize at every level
}


@pytest.mark.parametrize("engine", ["fp32", "bf16"])
@pytest.mark.parametrize("level", [3, 2, 1])
@pytest.mark.parametrize("size", list(SIZES))
def test_fusion_other_image_sizes(size, level, engine, monkeypatch):
    monkeypatch.setitem(synth.GEOMETRIES, size, SIZES[size])
    m, sd = module(level, engine)
    C, _, max_res, _ = synth.LEVELS[level]
    dt = DTYPES[engine]
    B = 3
    inp = synth.make_inputs(size, B, seed=6, levels=(level,))
    x = inp[f"x{level}"].to(dt)
    feat1 = randn(B, 64, 16, C, seed=level).to(dt)
    torch.manual_seed(13)
    with torch.no_grad():
        out = m(x.to(DEV), feat1.to(DEV), rect_data=inp["rect_data"], mask=inp["mask"].to(DEV), patch_info=inp["patch_info"],
                rgb=None)
    torch.cuda.synchronize()
    torch.manual_seed(13)
    ref = O.transformer_fusion(sd, synth.COMBINE1_LAYERS, max_res, x.double(), feat1.double(), inp["mask"], inp["patch_info"])
    H, W = x.shape[2:]
    regs = {**frame_regions(B, H, W), **tile_regions(B, H, W)}
    judge(out.permute(0, 2, 3, 1), ref.permute(0, 2, 3, 1), B, H, W, regs, "fusion", level, engine, f"fusion {size} L{level} {engine}")

