"""Training step of the path (BASELINE config 5): train-mode forward + backward through libcfp's fp32 training
kernels (``csrc/k_train.cu`` behind the ``cfp_tr_*`` entry points of include/cfp.h).

The reference trains these modules with autograd in fp32 (``train.py:96-135``; BatchNorm on per-replica batch statistics
under ``nn.DataParallel``, ``train.py:45``).  Here every op of the forward and of the backward is a libcfp kernel; this file
only sequences them - in the order of the closed-form backward (DESIGN.md section 8) - and owns the memory.
``torch.autograd.Function`` wrappers make the modules differentiable drop-ins: ``loss.backward()`` reaches the same
parameters the reference's autograd reaches, and the parameters the reference never uses keep ``grad is None``.

Built (SURVEY.md 8 / VERDICT r1 item 4): the histogram encoder (``HistogramEncoder``), LKPM (``Block14``) and - as a
sequence of primitive kernels ordered by ``cfpnet_b200/train_seq.py`` (``CudaOps`` / ``FusionTrainFn`` below) - a whole
``TransformerFusion`` call: hist2image, DAPM (attention + the two 3x3 convs with train-mode BatchNorm), LKPM, LSA, GSA.
Not served in training: the bilinear-resize branch of the zone canvas (fusion.py:141,146), ``--no_skip_inside``.
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, List, Tuple

import torch

from . import _lib
from .packing import PackCache

BN_EPS, BN_MOMENTUM = 1e-5, 0.1          # nn.BatchNorm defaults (encoder.py:10-12, convnext.py:39, transformer.py:198-200)
LKPM_LN_EPS = 1e-6                       # convnext.py:31


def _p(t):
    return 0 if t is None else t.data_ptr()


def _st():
    return _lib.stream_ptr()


def _f32c(t: torch.Tensor) -> torch.Tensor:
    t = t.detach()
    return t if (t.dtype == torch.float32 and t.is_contiguous()) else t.float().contiguous()


# ---------------------------------------------------------------------------------------------- op wrappers
def linear_fwd(x: torch.Tensor, w: torch.Tensor, bias) -> torch.Tensor:
    """x [R,K] @ w[N,K]^T + bias -> [R,N]"""
    R, K = x.shape
    N = w.shape[0]
    y = torch.empty(R, N, device=x.device, dtype=torch.float32)
    _lib.call("cfp_tr_gemm", x.data_ptr(), K, 1, w.data_ptr(), 1, K, y.data_ptr(), N, R, N, K, _p(bias), 0, _st())
    return y


def linear_dx(dy: torch.Tensor, w: torch.Tensor) -> torch.Tensor:
    """dy [R,N] @ w[N,K] -> [R,K]"""
    R, N = dy.shape
    K = w.shape[1]
    dx = torch.empty(R, K, device=dy.device, dtype=torch.float32)
    _lib.call("cfp_tr_gemm", dy.data_ptr(), N, 1, w.data_ptr(), K, 1, dx.data_ptr(), K, R, K, N, 0, 0, _st())
    return dx


def linear_dw(dy: torch.Tensor, x: torch.Tensor) -> torch.Tensor:
    """dy [R,N]^T @ x [R,K] -> [N,K]: the reduction over all rows of the batch."""
    R, N = dy.shape
    K = x.shape[1]
    dw = torch.empty(N, K, device=dy.device, dtype=torch.float32)
    _lib.call("cfp_tr_gemm", dy.data_ptr(), 1, N, x.data_ptr(), K, 1, dw.data_ptr(), K, N, K, R, 0, 0, _st())
    return dw


def colsum(x: torch.Tensor) -> torch.Tensor:
    R, Cc = x.shape
    out = torch.empty(Cc, device=x.device, dtype=torch.float32)
    _lib.call("cfp_tr_colsum", x.data_ptr(), out.data_ptr(), R, Cc, _st())
    return out


def bn_train_fwd(x: torch.Tensor, bn, relu: bool) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    """Train-mode BatchNorm of a [R,C] map (+ ReLU); updates bn.running_* / num_batches_tracked in place.
    Returns (y, mean, rstd)."""
    R, Cc = x.shape
    dev = x.device
    mean = torch.empty(Cc, device=dev, dtype=torch.float32)
    rstd = torch.empty(Cc, device=dev, dtype=torch.float32)
    scratch = torch.empty(2 * Cc, device=dev, dtype=torch.float32)
    rm, rv = bn.running_mean, bn.running_var
    if rm is not None and (rm.dtype != torch.float32 or not rm.is_contiguous()):
        raise _lib.CfpError("training runs in fp32: BatchNorm buffers must be contiguous float32")
    momentum = BN_MOMENTUM if bn.momentum is None else float(bn.momentum)
    _lib.call("cfp_tr_bn_stats", x.data_ptr(), R, Cc, float(bn.eps), momentum, mean.data_ptr(), rstd.data_ptr(),
              _p(rm), _p(rv), scratch.data_ptr(), _st())
    if bn.num_batches_tracked is not None:
        bn.num_batches_tracked.add_(1)
    y = torch.empty_like(x)
    _lib.call("cfp_tr_bn_apply", x.data_ptr(), mean.data_ptr(), rstd.data_ptr(), _f32c(bn.weight).data_ptr(),
              _f32c(bn.bias).data_ptr(), y.data_ptr(), R, Cc, int(relu), _st())
    return y, mean, rstd


def bn_train_bwd(dy, x, mean, rstd, bn, relu: bool):
    R, Cc = x.shape
    dx = torch.empty_like(x)
    dg = torch.empty(Cc, device=x.device, dtype=torch.float32)
    db = torch.empty(Cc, device=x.device, dtype=torch.float32)
    _lib.call("cfp_tr_bn_bwd", dy.data_ptr(), x.data_ptr(), mean.data_ptr(), rstd.data_ptr(), _f32c(bn.weight).data_ptr(),
              _f32c(bn.bias).data_ptr(), dx.data_ptr(), dg.data_ptr(), db.data_ptr(), R, Cc, int(relu), _st())
    return dx, dg, db


def ln_fwd(x, g, b, eps):
    R, Cc = x.shape
    y = torch.empty_like(x)
    _lib.call("cfp_tr_ln_fwd", x.data_ptr(), g.data_ptr(), b.data_ptr(), y.data_ptr(), R, Cc, float(eps), _st())
    return y


def ln_bwd(x, g, dy, eps):
    R, Cc = x.shape
    dx = torch.empty_like(x)
    dg = torch.empty(Cc, device=x.device, dtype=torch.float32)
    db = torch.empty(Cc, device=x.device, dtype=torch.float32)
    _lib.call("cfp_tr_ln_bwd", x.data_ptr(), g.data_ptr(), dy.data_ptr(), dx.data_ptr(), dg.data_ptr(), db.data_ptr(),
              R, Cc, float(eps), _st())
    return dx, dg, db


EW_ADD, EW_RELU_MASK, EW_GELU, EW_GELU_GRAD, EW_RELU, EW_ELU1_GRAD = range(6)


def ew(a, b, op, out=None):
    out = torch.empty_like(a) if out is None else out
    _lib.call("cfp_tr_ew", a.data_ptr(), _p(b), out.data_ptr(), a.numel(), op, _st())
    return out


def dwconv(x_tok, B, H, W, Cc, k, taps_t, shift, relu=False):
    out = torch.empty_like(x_tok)
    _lib.call("cfp_tr_dwconv", x_tok.data_ptr(), out.data_ptr(), B, H, W, Cc, k, taps_t.data_ptr(), shift.data_ptr(),
              int(relu), _st())
    return out


def dwconv_wgrad(x_tok, dy_tok, B, H, W, Cc, k):
    dw = torch.empty(Cc, k, k, device=x_tok.device, dtype=torch.float32)
    _lib.call("cfp_tr_dwconv_wgrad", x_tok.data_ptr(), dy_tok.data_ptr(), dw.data_ptr(), B, H, W, Cc, k, _st())
    return dw


# ---------------------------------------------------------------------------------------------- histogram encoder
def _hist_stages(mod):
    for ex in (mod.hist_extractor1, mod.hist_extractor2, mod.hist_extractor3):
        pe = ex.pointnet_encoder
        for conv, bn in ((pe.conv1, pe.bn1), (pe.conv2, pe.bn2), (pe.conv3, pe.bn3)):
            yield conv, bn


def hist_encoder_train_fwd(mod, hist_rows: torch.Tensor):
    """hist_rows [R,1] fp32 -> ([a3 [R,32], a6 [R,64], a9 [R,128]], saved).  encoder.py:17-24,31-35,45-50 in train mode."""
    a = hist_rows
    saved = []
    outs = []
    for i, (conv, bn) in enumerate(_hist_stages(mod)):
        w = _f32c(conv.weight)[:, :, 0].contiguous()
        y0 = linear_fwd(a, w, _f32c(conv.bias))
        y1, mean, rstd = bn_train_fwd(y0, bn, relu=True)
        saved.append((a, w, y0, mean, rstd))
        a = y1
        if i % 3 == 2:
            outs.append(a)
    return outs, saved


def hist_encoder_train_bwd(mod, saved, douts: List[torch.Tensor]):
    """Cotangents of the three outputs (None = unused) -> (dhist_rows [R,1], grads in parameter order of the stages)."""
    stages = list(_hist_stages(mod))
    grads: Dict[int, Tuple[torch.Tensor, ...]] = {}
    d = None
    for i in reversed(range(9)):
        if i % 3 == 2 and douts[i // 3] is not None:
            d = douts[i // 3] if d is None else ew(d, douts[i // 3], EW_ADD)
        if d is None:
            continue
        a_in, w, y0, mean, rstd = saved[i]
        _conv, bn = stages[i]
        dy0, dg, db = bn_train_bwd(d, y0, mean, rstd, bn, relu=True)
        gb = colsum(dy0)
        gw = linear_dw(dy0, a_in).unsqueeze(-1)
        grads[i] = (gw, gb, dg, db)
        d = linear_dx(dy0, w)
    return d, grads


class HistEncoderTrainFn(torch.autograd.Function):
    """forward(mod, hist [B,Z,S,1], *parameters in mod.parameters() order) -> (f32, f64, f128)."""

    @staticmethod
    def forward(ctx, mod, hist, *params):
        B, Z, S, _ = hist.shape
        rows = _f32c(hist).reshape(-1, 1)
        with torch.cuda.device(hist.device):
            outs, saved = hist_encoder_train_fwd(mod, rows)
        ctx.mod, ctx.saved, ctx.shape = mod, saved, (B, Z, S)
        ctx.set_materialize_grads(False)          # an unused output arrives as None, not as a zero map: its extractor is skipped
        return tuple(o.view(B, Z, S, -1) for o in outs)

    @staticmethod
    def backward(ctx, *douts):
        mod = ctx.mod
        B, Z, S = ctx.shape
        ds = [None if d is None else _f32c(d).reshape(B * Z * S, -1) for d in douts]
        with torch.cuda.device(ctx.saved[0][0].device):
            dhist, grads = hist_encoder_train_bwd(mod, ctx.saved, ds)
        by_param = {}
        for i, (conv, bn) in enumerate(_hist_stages(mod)):
            if i in grads:
                gw, gb, dg, db = grads[i]
                by_param[id(conv.weight)], by_param[id(conv.bias)] = gw, gb
                by_param[id(bn.weight)], by_param[id(bn.bias)] = dg, db
        pg = tuple(by_param.get(id(p)) for p in mod.parameters())
        return (None, None if dhist is None else dhist.view(B, Z, S, 1)) + pg


# ---------------------------------------------------------------------------------------------- LKPM (Block14)
def lkpm_train_fwd(blk, x_tok: torch.Tensor, B: int, H: int, W: int):
    """Block14.forward in train mode on a token-major map [B*H*W, C] (convnext.py:42-58): returns (out, saved)."""
    Cc = x_tok.shape[1]
    k = blk.dwconv2.kernel_size[0]
    taps = _f32c(blk.dwconv2.weight)[:, 0]                                   # [C,k,k]
    taps_t = taps.permute(1, 2, 0).reshape(k * k, Cc).contiguous()
    y0 = dwconv(x_tok, B, H, W, Cc, k, taps_t, _f32c(blk.dwconv2.bias))
    y2, mean, rstd = bn_train_fwd(y0, blk.bn1, relu=True)
    y3 = ln_fwd(y2, _f32c(blk.norm.weight), _f32c(blk.norm.bias), blk.norm.eps)
    w1, w2 = _f32c(blk.pwconv1.weight), _f32c(blk.pwconv2.weight)
    h0 = linear_fwd(y3, w1, _f32c(blk.pwconv1.bias))
    h = ew(h0, None, EW_GELU)
    out = linear_fwd(h, w2, _f32c(blk.pwconv2.bias))
    ew(out, x_tok, EW_ADD, out=out)
    # kept for the backward: the layer input, the pre-BN conv output with its statistics and the MLP pre-activation;
    # y2 / y3 / h are recomputed (elementwise passes)
    return out, (x_tok, y0, mean, rstd, h0, taps)


def lkpm_train_bwd(blk, saved, dout: torch.Tensor, B: int, H: int, W: int):
    """Returns (dx_tok, {parameter: gradient}) - the closed-form backward of DESIGN.md section 8, op by op."""
    x_tok, y0, mean, rstd, h0, taps = saved
    Cc = x_tok.shape[1]
    k = taps.shape[-1]
    R = x_tok.shape[0]
    bn = blk.bn1
    g_w, b_w = _f32c(bn.weight), _f32c(bn.bias)
    y2 = torch.empty_like(y0)
    _lib.call("cfp_tr_bn_apply", y0.data_ptr(), mean.data_ptr(), rstd.data_ptr(), g_w.data_ptr(), b_w.data_ptr(),
              y2.data_ptr(), R, Cc, 1, _st())
    ln_g, ln_b = _f32c(blk.norm.weight), _f32c(blk.norm.bias)
    y3 = ln_fwd(y2, ln_g, ln_b, blk.norm.eps)
    h = ew(h0, None, EW_GELU)
    w1, w2 = _f32c(blk.pwconv1.weight), _f32c(blk.pwconv2.weight)
    grads = {}
    grads[blk.pwconv2.bias] = colsum(dout)
    grads[blk.pwconv2.weight] = linear_dw(dout, h)
    dh0 = ew(linear_dx(dout, w2), h0, EW_GELU_GRAD)
    grads[blk.pwconv1.bias] = colsum(dh0)
    grads[blk.pwconv1.weight] = linear_dw(dh0, y3)
    dy2, grads[blk.norm.weight], grads[blk.norm.bias] = ln_bwd(y2, ln_g, linear_dx(dh0, w1), blk.norm.eps)
    dy0, grads[bn.weight], grads[bn.bias] = bn_train_bwd(dy2, y0, mean, rstd, bn, relu=True)
    grads[blk.dwconv2.bias] = colsum(dy0)
    grads[blk.dwconv2.weight] = dwconv_wgrad(x_tok, dy0, B, H, W, Cc, k).unsqueeze(1)
    flipped_t = torch.flip(taps, dims=(1, 2)).permute(1, 2, 0).reshape(k * k, Cc).contiguous()
    dm = dwconv(dy0, B, H, W, Cc, k, flipped_t, torch.zeros(Cc, device=x_tok.device, dtype=torch.float32))
    ew(dm, dout, EW_ADD, out=dm)
    return dm, grads


def _nchw_to_tokens(x: torch.Tensor) -> torch.Tensor:
    B, Cc, H, W = x.shape
    tok = torch.empty(B * H * W, Cc, device=x.device, dtype=torch.float32)
    zero_pos = torch.zeros(H * W, Cc, device=x.device, dtype=torch.float32)
    _lib.call("cfp_posenc_tokens_fwd", x.data_ptr(), zero_pos.data_ptr(), tok.data_ptr(), B, Cc, H, W, H, W, 0, 0, None,
              _lib.CFP_F32, _st())
    return tok


def _tokens_to_nchw(tok: torch.Tensor, B, Cc, H, W) -> torch.Tensor:
    out = torch.empty(B, Cc, H, W, device=tok.device, dtype=torch.float32)
    _lib.call("cfp_tokens_to_nchw", tok.data_ptr(), out.data_ptr(), B, Cc, H, W, _lib.CFP_F32, _st())
    return out


class LkpmTrainFn(torch.autograd.Function):
    """forward(blk, x [B,C,H,W], *parameters in blk.parameters() order) -> [B,C,H,W]  (Block14.forward, convnext.py:42-58)."""

    @staticmethod
    def forward(ctx, blk, x, *params):
        B, Cc, H, W = x.shape
        with torch.cuda.device(x.device):
            tok = _nchw_to_tokens(_f32c(x))
            out, saved = lkpm_train_fwd(blk, tok, B, H, W)
            res = _tokens_to_nchw(out, B, Cc, H, W)
        ctx.blk, ctx.saved, ctx.shape = blk, saved, (B, Cc, H, W)
        return res

    @staticmethod
    def backward(ctx, dout):
        blk = ctx.blk
        B, Cc, H, W = ctx.shape
        with torch.cuda.device(dout.device):
            d_tok = _nchw_to_tokens(_f32c(dout))
            dx_tok, grads = lkpm_train_bwd(blk, ctx.saved, d_tok, B, H, W)
            dx = _tokens_to_nchw(dx_tok, B, Cc, H, W)
        by_id = {id(p): g for p, g in grads.items()}
        pg = tuple(None if id(p) not in by_id else by_id[id(p)].reshape(p.shape) for p in blk.parameters())
        return (None, dx) + pg


# ---------------------------------------------------------------------------------------------- TransformerFusion in train mode
EW_ELU1, EW_NEG_DIV = 6, 7
_EW_CODES = {"add": EW_ADD, "relu": EW_RELU, "relu_mask": EW_RELU_MASK, "elu1": EW_ELU1, "elu1_grad_mul": EW_ELU1_GRAD,
             "neg_div": EW_NEG_DIV}
ROW_MUL, ROW_DIV, ROW_AXPY, ROW_GROUP_ADD, ROW_GROUP_SCALE = range(5)


class CudaOps:
    """The primitive ops ``cfpnet_b200/train_seq.py`` sequences, each one or two libcfp kernels on fp32 token-major
    ``[rows, C]`` maps (``cfp_tr_*``, include/cfp.h).  Same method names and semantics as the plain-torch stand-in the CPU
    test of the sequencing uses (tests/torch_ops.py); tests/test_gpu_train_fusion.py holds this class, through the same
    sequencing, to the reference's own ``.train()`` output and gradients."""

    # ---- dense
    def linear(self, x, w, bias=None, acc=None):
        x, w = _f32c(x), _f32c(w)
        R, K = x.shape
        N = w.shape[0]
        y = torch.empty(R, N, device=x.device, dtype=torch.float32) if acc is None else acc
        _lib.call("cfp_tr_gemm", x.data_ptr(), K, 1, w.data_ptr(), 1, K, y.data_ptr(), N, R, N, K,
                  _p(None if bias is None else _f32c(bias)), int(acc is not None), _st())
        return y

    def linear_dx(self, dy, w):
        return linear_dx(_f32c(dy), _f32c(w))

    def linear_dw(self, dy, x):
        return linear_dw(_f32c(dy), _f32c(x))

    def colsum(self, x):
        return colsum(_f32c(x))

    def ln_fwd(self, x, g, b, eps):
        return ln_fwd(x, _f32c(g), _f32c(b), eps)

    def ln_bwd(self, x, g, dy, eps):
        return ln_bwd(x, _f32c(g), _f32c(dy), eps)

    def bn_fwd(self, x, bn, relu):
        return bn_train_fwd(x, bn, relu)

    def bn_bwd(self, dy, x, mean, rstd, bn, relu):
        return bn_train_bwd(_f32c(dy), x, mean, rstd, bn, relu)

    def ew(self, a, b, op):
        return ew(_f32c(a), None if b is None else _f32c(b), _EW_CODES[op])

    # ---- linear attention (attention.py:31-49 and its closed-form backward)
    def attn_reduce(self, A, Bm, w, G, R, nh):
        Cc = A.shape[1]
        d = Cc // nh
        KV = torch.empty(G, nh, d, d, device=A.device, dtype=torch.float32)
        As = torch.empty(G, Cc, device=A.device, dtype=torch.float32)
        _lib.call("cfp_tr_attn_reduce", A.data_ptr(), Bm.data_ptr(), _p(w), KV.data_ptr(), As.data_ptr(), G, R, Cc, nh, _st())
        return KV, As

    def attn_apply(self, X, KV, G, R, nh, transpose):
        out = torch.empty_like(X)
        _lib.call("cfp_tr_attn_apply", X.data_ptr(), KV.data_ptr(), out.data_ptr(), G, R, X.shape[1], nh, int(bool(transpose)), _st())
        return out

    def head_dot(self, a, b, nh, rows_per_group, eps):
        n, Cc = a.shape
        out = torch.empty(n, nh, device=a.device, dtype=torch.float32)
        _lib.call("cfp_tr_head_dot", a.data_ptr(), b.data_ptr(), out.data_ptr(), n, Cc, nh, int(rows_per_group), float(eps), _st())
        return out

    def _rowop(self, a, s, b, out, nh, rpg, op):
        n, Cc = a.shape
        _lib.call("cfp_tr_rowop", a.data_ptr(), _p(s), _p(b), out.data_ptr(), n, Cc, nh, int(rpg), op, _st())
        return out

    def head_scale(self, a, s, nh, divide):
        return self._rowop(a, s, None, torch.empty_like(a), nh, 0, ROW_DIV if divide else ROW_MUL)

    def head_axpy(self, out, s, b, nh, rows_per_group):
        self._rowop(out, s, b, out, nh, rows_per_group, ROW_AXPY)

    def group_add(self, out, b, rows_per_group):
        self._rowop(out, None, b, out, 1, rows_per_group, ROW_GROUP_ADD)

    def group_scale(self, x, m, rows_per_group):
        return self._rowop(x, None, _f32c(m), torch.empty_like(x), 1, rows_per_group, ROW_GROUP_SCALE)

    # ---- regrouping
    def gather_rows(self, src, idx):
        src = _f32c(src)
        out = torch.empty(idx.numel(), src.shape[1], device=src.device, dtype=torch.float32)
        _lib.call("cfp_tr_gather_rows", src.data_ptr(), idx.data_ptr(), out.data_ptr(), idx.numel(), src.shape[1], _st())
        return out

    def scatter_add_rows(self, src, idx, base):
        out = torch.empty_like(base)
        _lib.call("cfp_tr_scatter_add_rows", src.data_ptr(), idx.data_ptr(), base.data_ptr(), out.data_ptr(), idx.numel(),
                  base.shape[0], base.shape[1], _st())
        return out

    def zeros_like(self, t):
        return torch.zeros_like(t)

    def index_mod(self, n, S, device):
        return (torch.arange(n, dtype=torch.int64) % S).to(torch.int32).to(device)

    # ---- layout
    def posenc_tokens(self, x, pos, max_res, oy, ox):
        B, Cc, H, W = x.shape
        tok = torch.empty(B * H * W, Cc, device=x.device, dtype=torch.float32)
        _lib.call("cfp_posenc_tokens_fwd", _f32c(x).data_ptr(), _f32c(pos).data_ptr(), tok.data_ptr(), B, Cc, H, W,
                  int(max_res[0]), int(max_res[1]), int(oy), int(ox), None, _lib.CFP_F32, _st())
        return tok

    def nchw_to_tokens(self, x):
        return _nchw_to_tokens(_f32c(x))

    def tokens_to_nchw(self, t, B, Cc, H, W):
        return _tokens_to_nchw(t, B, Cc, H, W)

    # ---- LKPM (the GPU-tested sequencing above)
    def lkpm_fwd(self, blk, x_tok, B, H, W):
        return lkpm_train_fwd(blk, x_tok, B, H, W)

    def lkpm_bwd(self, blk, saved, d, B, H, W):
        dx, grads = lkpm_train_bwd(blk, saved, d, B, H, W)
        names = {id(p): n for n, p in blk.named_parameters()}
        return dx, {names[id(p)]: g.reshape(p.shape) for p, g in grads.items()}


class FusionTrainFn(torch.autograd.Function):
    """forward(mod, x [B,C,H,W], feat1 [B,Z,S,C], zmask [B*Z] float, indexer, oy, ox, *parameters in
    mod.named_parameters() order) -> [B,C,H,W]: ``TransformerFusion.forward`` (fusion.py:52-188) in train mode.  Forward
    and backward are the op sequences of ``train_seq`` run on libcfp kernels; BatchNorm uses batch statistics and updates
    its running buffers; parameters the reference's autograd never reaches get no gradient."""

    @staticmethod
    def forward(ctx, mod, x, feat1, zmask, ix, oy, ox, *params):
        from . import train_seq as TS
        ops = CudaOps()
        P = {n: _f32c(p) for n, p in mod.named_parameters()}
        with torch.cuda.device(x.device):
            out, saved = TS.fusion_fwd(ops, mod, P, _f32c(x), _f32c(feat1), zmask, ix, oy, ox)
        ctx.mod, ctx.P, ctx.saved, ctx.zmask, ctx.ix, ctx.crop, ctx.f1shape = mod, P, saved, zmask, ix, (oy, ox), tuple(feat1.shape)
        return out

    @staticmethod
    def backward(ctx, dout):
        from . import train_seq as TS
        mod = ctx.mod
        with torch.cuda.device(dout.device):
            dx, dfeat1, grads = TS.fusion_bwd(CudaOps(), mod, ctx.P, ctx.saved, ctx.zmask, ctx.ix, ctx.crop[0], ctx.crop[1],
                                              _f32c(dout), ctx.f1shape)
        pg = tuple(None if n not in grads else grads[n].reshape(p.shape) for n, p in mod.named_parameters())
        return (None, dx, dfeat1, None, None, None, None) + pg


# ---------------------------------------------------------------------------------------------- the step around the modules
class FlatTrainer:
    """The reference's training step around the path's modules (train.py:96-135), one process per GPU:

        zero_grad -> forward -> loss.backward() -> [gradient all-reduce over NCCL] -> clip_grad_norm_(0.1) -> AdamW.step()

    The reference runs ``nn.DataParallel`` (train.py:45: replicas per step, per-replica BatchNorm statistics, gradients
    summed onto GPU 0); here every rank owns a replica and the gradients are AVERAGED over ranks (the loss is a mean over
    the batch) by ONE all-reduce of one flat fp32 bucket:

    * the parameters that receive a gradient (found by the first backward; the reference registers parameters it never
      uses, which keep ``grad is None`` and are skipped by its optimizer too) are re-homed as views into one flat buffer,
      and their ``.grad`` as views into a second one, so autograd accumulates straight into the bucket: no gather copy
      before the collective, no scatter after it;
    * ``cfp_tr_sumsq`` + ``cfp_tr_adamw`` do the clip + update on the flat buffers, reading the clip coefficient from
      device memory - the step never synchronises with the host.

    ``lr_of(param) -> float`` maps a parameter to its group's learning rate (the reference uses lr / 10 for the image
    encoder and lr for everything else, train.py:75-76)."""

    def __init__(self, modules, lr=1e-4, weight_decay=0.1, betas=(0.9, 0.999), eps=1e-8, max_norm=0.1, group=None,
                 lr_of=None):
        self.modules = list(modules)
        self.lr, self.wd, self.betas, self.eps, self.max_norm = float(lr), float(weight_decay), betas, float(eps), float(max_norm)
        self.group, self.lr_of = group, lr_of
        self.step_count = 0
        self.flat_p = self.flat_g = None
        self.allreduce_bytes = 0

    def parameters(self):
        seen = set()
        for m in self.modules:
            for p in m.parameters():
                if id(p) not in seen:
                    seen.add(id(p))
                    yield p

    def _world(self):
        import torch.distributed as dist
        return dist.get_world_size(self.group) if dist.is_available() and dist.is_initialized() else 1

    def adopt(self):
        """Call after the FIRST backward: builds the flat buffers over the parameters that received a gradient."""
        used = [p for p in self.parameters() if p.grad is not None]
        if not used:
            raise _lib.CfpError("FlatTrainer.adopt: no parameter has a gradient; run one forward + backward first")
        dev = used[0].device
        for p in used:
            if p.dtype != torch.float32 or p.device != dev:
                raise _lib.CfpError("training runs in fp32 on one device per process")
        world = self._world()
        if world > 1:                       # the used set must be the same on every rank (a mismatch would pair different tensors)
            import torch.distributed as dist
            idx = [i for i, p in enumerate(self.parameters()) if p.grad is not None]
            s = torch.tensor([len(idx), sum(idx), sum(i * i for i in idx)], dtype=torch.int64, device=dev)
            both = torch.cat([s, -s])
            dist.all_reduce(both, op=dist.ReduceOp.MAX, group=self.group)
            if not torch.equal(both[:3], -both[3:]):
                raise RuntimeError("ranks disagree on which parameters received a gradient")
        n = sum(p.numel() for p in used)
        self.flat_p = torch.empty(n, device=dev, dtype=torch.float32)
        self.flat_g = torch.zeros(n, device=dev, dtype=torch.float32)
        self.flat_m = torch.zeros(n, device=dev, dtype=torch.float32)
        self.flat_v = torch.zeros(n, device=dev, dtype=torch.float32)
        # segments of equal learning rate, in flat order
        seg_end, seg_lr, off = [], [], 0
        with torch.no_grad():
            for p in used:
                k = p.numel()
                self.flat_p[off:off + k].copy_(p.detach().reshape(-1))
                self.flat_g[off:off + k].copy_(p.grad.reshape(-1))
                p.data = self.flat_p[off:off + k].view(p.shape)
                p.grad = self.flat_g[off:off + k].view(p.shape)
                lr = float(self.lr_of(p)) if self.lr_of else self.lr
                off += k
                if seg_lr and seg_lr[-1] == lr:
                    seg_end[-1] = off
                else:
                    seg_end.append(off)
                    seg_lr.append(lr)
        self.used = used
        self.seg_end = torch.tensor(seg_end, dtype=torch.int64, device=dev)
        self.seg_lr = torch.tensor(seg_lr, dtype=torch.float32, device=dev)
        self.sumsq = torch.zeros(1026, device=dev, dtype=torch.float32)      # CFP_SUMSQ_FLOATS: result, partials, ticket
        return n

    def zero_grad(self):
        if self.flat_g is None:
            for p in self.parameters():
                p.grad = None
        else:
            self.flat_g.zero_()

    def exchange(self):
        """Sum the gradient bucket over the ranks (NCCL all-reduce; the 1 / world lands in the update).  Returns bytes."""
        world = self._world()
        if world == 1:
            return 0
        import torch.distributed as dist
        dist.all_reduce(self.flat_g, op=dist.ReduceOp.SUM, group=self.group)
        self.allreduce_bytes = self.flat_g.numel() * 4
        return self.allreduce_bytes

    def update(self):
        """clip_grad_norm_(max_norm) + AdamW on the flat buffers (after exchange())."""
        if self.flat_g is None:
            self.adopt()
        self.step_count += 1
        scale = 1.0 / self._world()
        n = self.flat_g.numel()
        with torch.cuda.device(self.flat_g.device):
            if self.max_norm > 0:
                _lib.call("cfp_tr_sumsq", self.flat_g.data_ptr(), n, C.c_float(scale), self.sumsq.data_ptr(), _st())
            _lib.call("cfp_tr_adamw", self.flat_p.data_ptr(), self.flat_g.data_ptr(), self.flat_m.data_ptr(),
                      self.flat_v.data_ptr(), n, self.seg_end.data_ptr(), self.seg_lr.data_ptr(), int(self.seg_lr.numel()),
                      C.c_float(self.betas[0]), C.c_float(self.betas[1]), C.c_float(self.eps), C.c_float(self.wd),
                      self.step_count, C.c_float(scale), self.sumsq.data_ptr(), C.c_float(self.max_norm), _st())
        for m in self.modules:               # packed eval-mode weights of the modules are stale now (every engine's cache)
            for sub in m.modules():
                for cache in list(vars(sub).values()):
                    if isinstance(cache, PackCache):
                        cache.invalidate()
