"""Generate ``tests/golden/trainblk_*.npz`` from the REFERENCE modules in TRAIN mode (container only).

    python tools/make_golden_train_blocks.py

Per-module fixtures for the training kernels (the first vertical slice of BASELINE config 5): the reference's
``HistogramEncoder`` (encoder.py:6-50) and ``Block14`` (LKPM, convnext.py:16-58) are imported from /root/reference, put in
``.train()`` mode in float64, run forward + backward with ``L = sum(out * cotangent)`` (seeded N(0,1) cotangents), and the
outputs, input gradients, EVERY parameter gradient and the BatchNorm buffers after the step are stored (float32 copies;
maps above 200k elements as a seeded sample + per-(frame, channel) sums).  tests/test_gpu_train.py holds the CUDA training
kernels to them; tests/test_oracle_train_blocks.py pins the oracle's closed-form backward on the same files.
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from ref_import import import_reference  # noqa: E402
from cfpnet_b200 import synth  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")
SAMPLE_N, FULL_LIMIT = 32768, 200_000            # keeps every fixture file under 1 MB
ref = import_reference()


def load_double(mod, seed):
    shapes = {k: v.shape for k, v in mod.state_dict().items()}
    sd = synth.synthetic_state_dict(shapes, seed=seed)
    mod.load_state_dict({k: v.double() if v.is_floating_point() else v for k, v in sd.items()}, strict=True)
    return mod


def pack_map(rec, key, t):
    rec[key + "_shape"] = np.array(t.shape)
    if t.numel() <= FULL_LIMIT:
        rec[key] = t.to(torch.float32).numpy()
    else:
        idx = torch.randperm(t.numel(), generator=torch.Generator().manual_seed(1234))[:SAMPLE_N]
        rec[key + "_idx"] = idx.numpy().astype(np.int64)
        rec[key + "_sample"] = t.reshape(-1)[idx].to(torch.float32).numpy()
        rec[key + "_perchan"] = t.sum(dim=(2, 3)).to(torch.float32).numpy()


def rel(a, b):
    return float((a.double() - b.double()).norm() / b.double().norm().clamp_min(1e-300))


def pack_ref32(rec, mod64, mod32):
    """The reference's OWN float32 run of the same step against its float64 run, per parameter gradient: where that
    deviation is large the gradient is cancellation-dominated (e.g. the weight of a 1-input conv in front of a
    batch-statistics BatchNorm: mathematically ~0) and no fp32 implementation can match fp64 to 1e-3 there."""
    g64 = {n: p.grad for n, p in mod64.named_parameters() if p.grad is not None}
    for n, p in mod32.named_parameters():
        if p.grad is not None:
            rec["ref32err:" + n] = np.float64(rel(p.grad, g64[n]))


def pack_module(rec, mod):
    names, has = [], []
    for n, p in mod.named_parameters():
        names.append(n)
        has.append(p.grad is not None)
        if p.grad is not None:
            rec["grad:" + n] = p.grad.to(torch.float32).numpy()
    rec["param_names"], rec["param_has_grad"] = np.array(names), np.array(has)
    for n, b in mod.named_buffers():
        rec["buf:" + n] = b.detach().numpy()


def hist_case(batch=2):
    enc = load_double(ref["encoder"].HistogramEncoder().double(), 0).train()
    inp = synth.make_inputs("G416", batch, seed=1, levels=())
    hist = inp["hist_data"].double().requires_grad_(True)
    outs = enc(hist.unsqueeze(-1))
    g = torch.Generator().manual_seed(77)
    cts = [torch.randn(o.shape, generator=g, dtype=torch.float64) for o in outs]
    sum((o * c).sum() for o, c in zip(outs, cts)).backward()
    rec = {"grad_hist": hist.grad.to(torch.float32).numpy()}
    for c_, o in zip((32, 64, 128), outs):
        pack_map(rec, f"out{c_}", o.detach())
    pack_module(rec, enc)
    enc32 = load_double(ref["encoder"].HistogramEncoder().double(), 0).float().train()
    outs32 = enc32(inp["hist_data"].float().unsqueeze(-1))
    sum((o * c.float()).sum() for o, c in zip(outs32, cts)).backward()
    pack_ref32(rec, enc, enc32)
    np.savez_compressed(os.path.join(OUT, f"trainblk_hist_B{batch}.npz"), **rec)
    print("hist encoder", [tuple(o.shape) for o in outs], "|grad_hist|", float(hist.grad.norm()))


def lkpm_case(level, batch):
    C, _, _, k = synth.LEVELS[level]
    H, W = synth.level_hw("G416", level)
    blk = load_double(ref["convnext"].Block14(C, large_kernel=k).double(), 3).train()
    x = torch.randn(batch, C, H, W, generator=torch.Generator().manual_seed(5), dtype=torch.float64).requires_grad_(True)
    out = blk(x)
    ct = torch.randn(out.shape, generator=torch.Generator().manual_seed(78), dtype=torch.float64)
    (out * ct).sum().backward()
    rec = {"meta": np.array([str(level), str(batch), str(C), str(k), str(H), str(W)])}
    pack_map(rec, "out", out.detach())
    pack_map(rec, "grad_x", x.grad)
    pack_module(rec, blk)
    blk32 = load_double(ref["convnext"].Block14(C, large_kernel=k).double(), 3).float().train()
    (blk32(x.detach().float()) * ct.float()).sum().backward()
    pack_ref32(rec, blk, blk32)
    np.savez_compressed(os.path.join(OUT, f"trainblk_lkpm_L{level}_B{batch}.npz"), **rec)
    print(f"lkpm L{level}", tuple(out.shape), "|grad_x|", float(x.grad.norm()),
          "never used:", [n for n, p in blk.named_parameters() if p.grad is None])


if __name__ == "__main__":
    hist_case(2)
    lkpm_case(3, 2)
    lkpm_case(2, 2)
    lkpm_case(1, 1)
