"""Training kernels (BASELINE config 5, first vertical slice) against the REFERENCE's own train-mode forward + backward:
fixtures tests/golden/trainblk_*.npz come from the reference's HistogramEncoder / Block14 in .train() mode (float64,
tools/make_golden_train_blocks.py).  The CUDA path runs through the drop-in modules -> autograd Function ->
cfp_tr_* kernels (fp32).  Tolerance: rel-L2 <= 1e-3 per tensor (outputs, input gradients, every parameter gradient,
BatchNorm buffers after the step); parameters the reference never uses must keep grad None."""
import os

import numpy as np
import pytest
import torch

import cfpnet_b200
from cfpnet_b200 import synth
from helpers import GOLDEN, rel_l2

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
TOL = 1e-3


def load(mod, seed):
    mod.load_state_dict(synth.synthetic_state_dict({k: v.shape for k, v in mod.state_dict().items()}, seed=seed), strict=True)
    return mod.to(DEV).train()


def check_module(mod, z, what):
    names = [str(n) for n in z["param_names"]]
    has = dict(zip(names, [bool(v) for v in z["param_has_grad"]]))
    for n, p in mod.named_parameters():
        if not has[n]:
            assert p.grad is None, f"{what}: {n} is never used by the reference and must keep grad None"
            continue
        assert p.grad is not None, f"{what}: {n} received no gradient"
        want = torch.from_numpy(z["grad:" + n])
        assert p.grad.shape == want.shape
        err = rel_l2(p.grad, want)
        # a conv / linear bias in front of a batch-statistics BatchNorm has an exactly-zero gradient (the reference's
        # autograd leaves 1e-16 rounding noise there): compare those against the scale of the layer's weight gradient
        if float(want.norm()) < 1e-9 * max(1.0, float(p.grad.numel()) ** 0.5):
            assert float(p.grad.norm()) <= 1e-3 * float(z["grad:" + n.rsplit(".", 1)[0] + ".weight"].std() + 1e-30) * p.grad.numel() ** 0.5 + 1e-4, \
                f"{what}: {n} should be ~0, got |g| = {float(p.grad.norm()):.3e}"
            continue
        # cancellation-dominated gradients (a weight whose scale batch-statistics BatchNorm removes again: size eps/var of
        # its terms): the reference's own fp32 run misses its fp64 run by `ref32err` there - allow 10x that
        tol = max(TOL, 10.0 * float(z["ref32err:" + n]))
        assert err <= tol, f"{what}: grad {n} rel-L2 {err:.3e} (tolerance {tol:.1e})"
    for n, b in mod.named_buffers():
        want = torch.from_numpy(np.asarray(z["buf:" + n]))
        if want.dtype == torch.int64:
            assert int(b) == int(want), f"{what}: {n}"
        else:
            assert rel_l2(b, want) <= TOL, f"{what}: buffer {n} rel-L2 {rel_l2(b, want):.3e}"


def check_map(got, z, key, what):
    got = got.detach().double().cpu()
    assert tuple(got.shape) == tuple(int(v) for v in z[key + "_shape"])
    if key in z.files:
        err = rel_l2(got, torch.from_numpy(z[key]))
        assert err <= TOL, f"{what}: {key} rel-L2 {err:.3e}"
        return
    idx = torch.from_numpy(z[key + "_idx"])
    e1 = rel_l2(got.reshape(-1)[idx], torch.from_numpy(z[key + "_sample"]))
    e2 = rel_l2(got.sum(dim=(2, 3)), torch.from_numpy(z[key + "_perchan"]))
    assert e1 <= TOL and e2 <= TOL, f"{what}: {key} rel-L2 sample {e1:.3e} perchan {e2:.3e}"


def test_hist_encoder_train_step_matches_reference():
    z = np.load(os.path.join(GOLDEN, "trainblk_hist_B2.npz"))
    enc = load(cfpnet_b200.HistogramEncoder(), 0)
    inp = synth.make_inputs("G416", 2, seed=1, levels=())
    hist = inp["hist_data"].to(DEV).requires_grad_(True)
    outs = enc(hist.unsqueeze(-1))
    g = torch.Generator().manual_seed(77)
    cts = [torch.randn(o.shape, generator=g, dtype=torch.float64) for o in outs]
    sum((o * c.float().to(DEV)).sum() for o, c in zip(outs, cts)).backward()
    torch.cuda.synchronize()
    for c_, o in zip((32, 64, 128), outs):
        check_map(o, z, f"out{c_}", "hist encoder")
    assert rel_l2(hist.grad, torch.from_numpy(z["grad_hist"])) <= TOL
    check_module(enc, z, "hist encoder")


def test_hist_encoder_train_partial_cotangents():
    """Only the 64-channel output is used downstream: the third extractor gets no gradient at all (grad stays None), the
    first two do - what happens when a decoder level is frozen."""
    enc = load(cfpnet_b200.HistogramEncoder(), 0)
    inp = synth.make_inputs("G416", 1, seed=3, levels=())
    outs = enc(inp["hist_data"].to(DEV).unsqueeze(-1))
    outs[1].sum().backward()
    assert enc.hist_extractor3.pointnet_encoder.conv1.weight.grad is None
    assert enc.hist_extractor2.pointnet_encoder.conv3.weight.grad is not None
    assert enc.hist_extractor1.pointnet_encoder.conv1.weight.grad is not None


@pytest.mark.parametrize("level,batch", [(3, 2), (2, 2), (1, 1)])
def test_lkpm_train_step_matches_reference(level, batch):
    z = np.load(os.path.join(GOLDEN, f"trainblk_lkpm_L{level}_B{batch}.npz"))
    C, _, _, k = synth.LEVELS[level]
    H, W = synth.level_hw("G416", level)
    blk = load(cfpnet_b200.layers.Block14(C, large_kernel=k), 3)
    x = torch.randn(batch, C, H, W, generator=torch.Generator().manual_seed(5), dtype=torch.float64).float().to(DEV).requires_grad_(True)
    out = blk(x)
    ct = torch.randn(out.shape, generator=torch.Generator().manual_seed(78), dtype=torch.float64).float().to(DEV)
    (out * ct).sum().backward()
    torch.cuda.synchronize()
    check_map(out, z, "out", f"lkpm L{level}")
    check_map(x.grad, z, "grad_x", f"lkpm L{level}")
    check_module(blk, z, f"lkpm L{level}")


def test_training_kernels_against_torch_ops_on_ragged_shapes():
    """The building blocks on shapes that are not tile multiples, against plain fp64 torch ops on the same inputs."""
    from cfpnet_b200 import train as T
    g = torch.Generator().manual_seed(0)
    R, K, N = 1000, 40, 72
    x = torch.randn(R, K, generator=g).to(DEV)
    w = torch.randn(N, K, generator=g).to(DEV)
    b = torch.randn(N, generator=g).to(DEV)
    dy = torch.randn(R, N, generator=g).to(DEV)
    with torch.cuda.device(0):
        assert rel_l2(T.linear_fwd(x, w, b), x.double() @ w.double().t() + b.double()) <= 1e-5
        assert rel_l2(T.linear_dx(dy, w), dy.double() @ w.double()) <= 1e-5
        assert rel_l2(T.linear_dw(dy, x), dy.double().t() @ x.double()) <= 1e-5
        big = torch.randn(70000, 24, generator=g).to(DEV)                      # split-K path (atomics)
        bigy = torch.randn(70000, 36, generator=g).to(DEV)
        assert rel_l2(T.linear_dw(bigy, big), bigy.double().t() @ big.double()) <= 1e-5
        assert rel_l2(T.colsum(big), big.double().sum(0)) <= 1e-5
        gam, bet = (torch.rand(K, generator=g) + 0.5).to(DEV), torch.randn(K, generator=g).to(DEV)
        y = T.ln_fwd(x, gam, bet, 1e-5)
        xd = x.double().requires_grad_(True)
        gd, bd = gam.double().requires_grad_(True), bet.double().requires_grad_(True)
        yd = torch.nn.functional.layer_norm(xd, (K,), gd, bd, 1e-5)
        assert rel_l2(y, yd) <= 1e-5
        ct = torch.randn(R, K, generator=g).to(DEV)
        (yd * ct.double()).sum().backward()
        dx, dg, db = T.ln_bwd(x, gam, ct, 1e-5)
        assert rel_l2(dx, xd.grad) <= 1e-4 and rel_l2(dg, gd.grad) <= 1e-4 and rel_l2(db, bd.grad) <= 1e-4
