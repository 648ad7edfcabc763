"""Drop-in for the reference's ``TransformerFusion`` (``src/models/fusion.py:12-188``).

Same constructor signature, same ``forward(x, feat1, **kwargs)`` contract
(kwargs: ``rect_data``, ``mask``, ``patch_info``, ``rgb``), same parameter names
and shapes, same draws from torch's global CPU generator for the positional-
encoding crop.  Every tensor op of the reference's forward is replaced by
hand-written sm_100a kernels behind the C ABI of include/cfp.h; this file only
computes the host integers, owns the memory and sequences the launches.
"""
from __future__ import annotations

import ctypes as C
import math

import torch
import torch.nn as nn

from . import _lib
from .config import args
from .geometry import check_geometry, zone_geometry
from .layers import Combine1, LoFTREncoderLayer, TwinsTransformer
from .packing import PackCache, Packer, Scratch, host, relocate


class TransformerFusion(nn.Module):
    def __init__(self, embedding_dim, max_resolution, num_heads=4, large_kernel=None, patch_size=None):
        super().__init__()
        if num_heads != 4:
            raise NotImplementedError("libcfp serves the hist2image / DAPM layers with 4 heads (fusion.py:13)")
        self.zone_sample_num = args.zone_sample_num
        self.max_resolution = max_resolution
        self.embedding_dim = embedding_dim
        self.large_kernel = large_kernel if "combine1" in args.attention_layer else 0
        self.positional_encodings = nn.Parameter(
            torch.rand(max_resolution[0] * max_resolution[1], embedding_dim), requires_grad=True)
        self.positional_encodings2 = nn.Parameter(
            torch.rand(self.zone_sample_num, embedding_dim), requires_grad=True)
        nn.init.trunc_normal_(self.positional_encodings, std=0.2)
        nn.init.trunc_normal_(self.positional_encodings2, std=0.2)

        self.layer_names = list(args.attention_layer)
        self.ws = math.ceil(math.sqrt(math.sqrt(max_resolution[0] * max_resolution[1])))   # fusion.py:28
        layers = []
        for name in self.layer_names:
            if name == "image":
                layers.append(TwinsTransformer(embedding_dim, num_heads, ws=self.ws))
            elif name == "hist2image":
                layers.append(LoFTREncoderLayer(embedding_dim, num_heads))
            elif name == "combine1":
                layers.append(Combine1(embedding_dim, num_heads, large_kernel=large_kernel))
            else:
                raise NotImplementedError(name)           # fusion.py:37
        self.layers = nn.ModuleList(layers)
        self.conv_patch_size = 640 / self.max_resolution[1]
        self._cache = PackCache()
        self._scratch = Scratch()

    def _replicate_for_data_parallel(self):
        """``nn.DataParallel`` replicas copy ``__dict__`` shallowly: give each its own pack cache and scratch (the
        original's hold device-0 pointers) - replicas run concurrently, one thread per GPU (train.py:45)."""
        replica = super()._replicate_for_data_parallel()
        replica._cache = PackCache()
        replica._scratch = Scratch()
        return replica

    # ------------------------------------------------------------------ packing
    def _pack(self):
        """Weight structs of every layer + the two positional tables: packed on the host, one flat device buffer
        (``buf``), struct fields relocated to device pointers.  Returns (structs, pos ptr, pos2 ptr, buf)."""
        keep = Packer()
        packed = []
        for layer, name in zip(self.layers, self.layer_names):
            if name == "combine1":
                packed.append((layer.transformer_path.pack(keep), layer.large_kernel_path.pack(keep)))
            else:
                packed.append(layer.pack(keep))
        pos = keep.ref(host(self.positional_encodings).contiguous())
        pos2 = keep.ref(host(self.positional_encodings2).contiguous())
        buf = keep.upload(self.positional_encodings.device)
        base = buf.data_ptr()
        for w in packed:
            for s_ in (w if isinstance(w, tuple) else (w,)):
                relocate(s_, base)
        return packed, base + pos, base + pos2, buf


    def draw_crop(self, H: int, W: int):
        """(oy, ox) of the positional-encoding crop: the reference's draws from torch's global CPU generator, in its
        order (fusion.py:87-91); nothing is drawn along an axis the map fills."""
        if H > self.max_resolution[0] or W > self.max_resolution[1]:
            raise ValueError("feature map larger than the positional-encoding table")
        oy = ox = 0
        if H < self.max_resolution[0]:
            oy = int(torch.randint(0, self.max_resolution[0] - H + 1, [1]))
        if W < self.max_resolution[1]:
            ox = int(torch.randint(0, self.max_resolution[1] - W + 1, [1]))
        return oy, ox

    def _run_layers(self, packed, pos2, feat0, feat1, mask, B, H, W, D, S, cg, work, ws_bytes, code, st, emb_copy,
                    out_nchw=None) -> bool:
        """The layer list on the token-major map ``feat0`` [B, H*W, D] (in place), current stream.  With ``out_nchw`` (a
        contiguous [B, D, H, W] tensor) and an ``image`` layer last, that layer's last epilogue writes the NCHW result
        itself and True is returned; otherwise the result is in ``feat0`` (False)."""
        emb = feat0.clone() if emb_copy else feat0           # fusion.py:134-136: canvas cut from the first map
        last = len(self.layer_names) - 1
        for i, (w, name) in enumerate(zip(packed, self.layer_names)):
            if name == "image" and i == last and out_nchw is not None:
                _lib.call("cfp_twins_nchw_fwd", feat0.data_ptr(), out_nchw.data_ptr(), B, H, W, D, C.byref(w), work.data_ptr(),
                          ws_bytes, code, st)
                return True
            if name == "image":
                _lib.call("cfp_twins_fwd", feat0.data_ptr(), B, H, W, D, C.byref(w), work.data_ptr(), ws_bytes, code, st)
            elif name == "hist2image":
                _lib.call("cfp_d2i_fwd", feat0.data_ptr(), emb.data_ptr(), feat1.data_ptr(), pos2, mask.data_ptr(), B, H, W, D, S,
                          C.byref(cg), C.byref(w), int(bool(args.no_skip_inside)), work.data_ptr(), ws_bytes, code, st)
            else:   # combine1: DAPM then LKPM (transformer.py:270-273)
                dapm_w, lkpm_w = w
                _lib.call("cfp_dapm_fwd", feat0.data_ptr(), B, H, W, D, C.byref(cg), C.byref(dapm_w), work.data_ptr(), ws_bytes,
                          code, st)
                _lib.call("cfp_lkpm_fwd", feat0.data_ptr(), B, H, W, D, C.byref(lkpm_w), work.data_ptr(), ws_bytes, code, st)
        return False

    def _prepare(self, x, B, H, W, feat1, kwargs, check=None):
        """Set-up shared by ``forward`` and ``forward_tokens`` for the map ``x`` (its dtype selects the engine), in this order:
        the shape checks, the caller's own ``check()``, the positional-encoding draws, then the packed weights, feat1 and
        mask in the engine's types and the call's scratch.  Returns (pos, oy, ox, crop_dev, feat0, layers): ``crop_dev`` is
        the device crop buffer under a CUDA-graph capture (oy = ox = 0 then), else None; ``feat0`` is the [B, H*W, D] token
        map the caller fills; ``layers(st, out_nchw=None)`` runs the layer list on it (``_run_layers``)."""
        D, dt, dev = self.embedding_dim, x.dtype, x.device
        S = feat1.size(2)
        g = zone_geometry(kwargs["patch_info"], self.max_resolution[1], H, W)
        if any(n in ("hist2image", "combine1") for n in self.layer_names):
            check_geometry(g, H, W)
        if feat1.shape[0] != B or feat1.shape[1] != g.zone_num ** 2 or feat1.shape[3] != D:
            raise ValueError(f"feat1 {tuple(feat1.shape)} does not match B={B}, zones={g.zone_num ** 2}, D={D}")
        if S != self.positional_encodings2.shape[0]:     # the reference's `feat1 + positional_encodings2` fails to broadcast
            raise ValueError(f"feat1 carries {S} samples per zone, positional_encodings2 has {self.positional_encodings2.shape[0]}")
        if tuple(kwargs["mask"].shape) != (B, g.zone_num ** 2):
            raise ValueError(f"mask {tuple(kwargs['mask'].shape)} is not [B={B}, zones={g.zone_num ** 2}]")
        if check is not None:
            check()

        # positional-encoding crop: same draws, same order as fusion.py:87-91 (under a CUDA-graph capture the offsets live
        # in device memory and the replay wrapper makes the draws: FusionPath.make_graphed, pipeline.make_graphed_depth)
        crop_dev = self.__dict__.get("_crop_dev")
        oy, ox = (0, 0) if crop_dev is not None else self.draw_crop(H, W)

        packed, pos, pos2, _buf = self._cache.get(self, self._pack)
        feat1 = feat1.detach().to(dt).contiguous()
        mask = kwargs["mask"].to(device=dev, dtype=torch.uint8).contiguous()
        cg = _lib.CfpGeom.from_geometry(g)
        emb_copy = (not args.change_embedding) and "hist2image" in self.layer_names
        code = _lib.dtype_code(dt)
        ws_bytes = _lib.load().cfp_workspace_bytes(B, H, W, D, self.ws, self.large_kernel or 0, code, C.byref(cg))
        # scratch (workspace + token map) is owned by the module and reused across calls: stream order
        # makes that safe for back-to-back forwards on one stream, and it keeps hundreds of MB of
        # per-call allocations (cudaMalloc stalls once several streams are in play) off the hot path.
        # One module instance must not run on two streams at once (replicas own their scratch).
        work, feat0 = self._scratch.get(
            dev.index, (dt, B, H, W), lambda t: t[0].numel() >= ws_bytes,
            lambda: (torch.empty(ws_bytes, device=dev, dtype=torch.uint8), torch.empty(B, H * W, D, device=dev, dtype=dt)))

        def layers(st, out_nchw=None):
            return self._run_layers(packed, pos2, feat0, feat1, mask, B, H, W, D, S, cg, work, ws_bytes, code, st, emb_copy,
                                    out_nchw=out_nchw)
        return pos, oy, ox, crop_dev, feat0, layers

    def forward_tokens(self, x_tok, x_pitch, B, H, W, feat1, out_tok, out_pitch, out_coff, **kwargs):
        """The same call for a caller that holds its maps channels-last (cfpnet_b200.decoder): ``x_tok`` is a
        [B, H, W, x_pitch] buffer whose first ``embedding_dim`` channels are x; the result is written into channels
        [out_coff, out_coff + embedding_dim) of ``out_tok`` [B, H, W, out_pitch] - the ``torch.cat([x_d, x_d_fused])`` of
        decoder.py:112,117,122 without a transposed or concatenated copy.  Same positional-encoding draws as forward().
        Both maps bf16 run the tensor-core engine, both fp32 the exact fp32 engine (the module's parameters in fp32)."""
        if self.training:
            raise NotImplementedError("libcfp serves eval-mode BatchNorm only for the attention layers")
        _lib.require_cuda(x_tok, "x_tok")
        D = self.embedding_dim
        dt = x_tok.dtype
        if dt not in (torch.bfloat16, torch.float32) or out_tok.dtype != dt:
            raise ValueError(f"forward_tokens needs x_tok and out_tok both bf16 or both fp32 (got {x_tok.dtype} and {out_tok.dtype})")
        pos, oy, ox, crop_dev, feat0, layers = self._prepare(x_tok, B, H, W, feat1, kwargs)
        code = _lib.dtype_code(dt)
        with torch.cuda.device(x_tok.device):
            st = _lib.stream_ptr()
            _lib.call("cfp_posenc_tokens_nhwc_fwd", x_tok.data_ptr(), x_pitch, pos, feat0.data_ptr(), B, D, H, W,
                      self.max_resolution[0], self.max_resolution[1], oy, ox, _lib.ptr(crop_dev), code, st)
            layers(st)
            _lib.call("cfp_copy_channels", feat0.data_ptr(), D, out_tok.data_ptr(), out_pitch, out_coff, D, B * H * W, code, st)
        return out_tok

    # ------------------------------------------------------------------ forward
    def _forward_train(self, x, feat1, **kwargs):
        """Train mode (BASELINE config 5; reference train.py:96-135 differentiates fusion.py:52-188 with autograd): fp32,
        BatchNorm on batch statistics, differentiable w.r.t. x, feat1 and every parameter the reference's autograd
        reaches - cfpnet_b200/train.py (FusionTrainFn) runs the op sequence of cfpnet_b200/train_seq.py on libcfp kernels."""
        from . import train as T
        from . import train_seq as TS
        _lib.require_cuda(x, "x")
        B, D, H, W = x.shape
        if D != self.embedding_dim:
            raise ValueError(f"x has {D} channels, module was built for {self.embedding_dim}")
        if any(p.dtype != torch.float32 for p in self.parameters()):
            raise _lib.CfpError("training runs in fp32 (as the reference trains): cast the module with .float()")
        g = zone_geometry(kwargs["patch_info"], self.max_resolution[1], H, W)
        if any(n in ("hist2image", "combine1") for n in self.layer_names):
            check_geometry(g, H, W)
        if g.interpolate or args.no_skip_inside or not args.change_embedding:
            raise NotImplementedError("training serves the no-resize zone canvas with change_embedding (the reference's "
                                      "training geometry); the resize branch / --no_skip_inside are eval-only here")
        S = feat1.size(2)
        if feat1.shape[0] != B or feat1.shape[1] != g.zone_num ** 2 or feat1.shape[3] != D or S != self.positional_encodings2.shape[0]:
            raise ValueError(f"feat1 {tuple(feat1.shape)} does not match B={B}, zones={g.zone_num ** 2}, D={D}")
        if tuple(kwargs["mask"].shape) != (B, g.zone_num ** 2):
            raise ValueError(f"mask {tuple(kwargs['mask'].shape)} is not [B={B}, zones={g.zone_num ** 2}]")
        oy, ox = self.draw_crop(H, W)
        key = (B, H, W, g, str(x.device))             # the index vectors depend on the shapes and the zone geometry only
        cache = self.__dict__.setdefault("_train_ix", {})
        if key not in cache:
            cache.clear()
            cache[key] = TS.Indexer(B, H, W, g, self.ws, x.device)
        zmask = kwargs["mask"].to(device=x.device, dtype=torch.float32).reshape(-1).contiguous()
        params = [p for _, p in self.named_parameters()]
        return T.FusionTrainFn.apply(self, x, feat1, zmask, cache[key], oy, ox, *params)

    def forward(self, x, feat1, **kwargs):
        if self.training:
            return self._forward_train(x, feat1, **kwargs)
        _lib.require_cuda(x, "x")
        B, D, H, W = x.shape
        if D != self.embedding_dim:
            raise ValueError(f"x has {D} channels, module was built for {self.embedding_dim}")
        dt = x.dtype
        code = _lib.dtype_code(dt)

        def refuse_grad():
            if torch.is_grad_enabled() and (x.requires_grad or feat1.requires_grad):
                raise RuntimeError("TransformerFusion (libcfp, eval mode) returns a tensor without autograd history: an input "
                                   "that requires grad would have its gradient cut silently; call under torch.no_grad() or "
                                   "detach the inputs")

        pos, oy, ox, crop_dev, feat0, layers = self._prepare(x, B, H, W, feat1, kwargs, check=refuse_grad)
        dev = x.device
        x = x.detach().contiguous()
        out = kwargs.get("out")                  # optional caller-provided result buffer (same shape/dtype)
        if out is None:
            out = torch.empty(B, D, H, W, device=dev, dtype=dt)
        elif out.shape != x.shape or out.dtype != dt or out.device != dev or not out.is_contiguous():
            raise ValueError("out= must be a contiguous tensor shaped and typed like x")

        with torch.cuda.device(dev):
            st = _lib.stream_ptr()
            _lib.call("cfp_posenc_tokens_fwd", x.data_ptr(), pos, feat0.data_ptr(), B, D, H, W,
                      self.max_resolution[0], self.max_resolution[1], oy, ox, _lib.ptr(crop_dev), code, st)
            if not layers(st, out_nchw=out):
                _lib.call("cfp_tokens_to_nchw", feat0.data_ptr(), out.data_ptr(), B, D, H, W, code, st)
        return out
