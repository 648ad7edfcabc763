"""Shared test plumbing: golden fixtures, synthetic cases, error metrics."""
import json
import os

import numpy as np
import torch

from cfpnet_b200 import synth

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

FUSION_CASES = [
    "G416_L3_B2", "G416_L2_B1", "G416_L1_B1", "G480_L3_B1", "G480pad_L3_B1", "G480pad_L2_B1",
    "G416_L3_B1_baseline", "G416_L3_B1_noskip", "G416_L3_B1_keepemb",
    # round 2: every shape a bench configuration runs (BASELINE.json configs[1] / [3]) at every level it touches
    "G480_L2_B1", "G480_L1_B1", "G480pad_L1_B1", "G416_L2_B1_baseline", "G416_L1_B1_baseline", "G416_L3_B16_baseline",
]
# 6x6 zones of 64 px - the reference's training layout (--train_zone_num 6).  Fixtures from the reference; oracle,
# geometry and (since the workspace-size fix, profiles/r1t_z6_gpu_check.log) the CUDA path are held to them.
FUSION_CASES_Z6 = ["G416z6_L3_B2", "G416z6_L2_B1", "G416z6_L1_B1"]


def rel_l2(a: torch.Tensor, b: torch.Tensor) -> float:
    a, b = a.double().cpu(), b.double().cpu()
    return float((a - b).norm() / b.norm().clamp_min(1e-30))


MIN_REGION = 16          # regions with fewer tokens are reported but not bounded: their rel-L2 is too noisy to hold to a ratio


def region_errors(out: torch.Tensor, ref: torch.Tensor, regions: dict, bulk=None) -> dict:
    """Where an error sits.  ``out`` / ``ref``: [B, H, W, C] maps; ``regions``: name -> bool token mask [B, H, W];
    ``bulk``: the tokens the layer actually changes (all tokens when None).

    Returns ``bulk`` (rel-L2 over the bulk tokens, all channels), ``regions`` (name -> (rel-L2 over the region's tokens,
    token count)), ``token`` (the largest ||out_t - ref_t|| over the bulk, divided by the RMS token norm of ``ref`` in the
    token's frame) with its place ``token_at`` = (frame, row, column), and ``ratio`` (the largest region error over the
    bulk error among regions of at least ``MIN_REGION`` tokens).  A defect confined to a few percent of the tokens moves a
    whole-map rel-L2 by little; the same defect dominates its own region and its own tokens."""
    o, r = out.detach().double().cpu(), ref.detach().double().cpu()
    e2 = (o - r).pow(2).sum(-1)                                  # [B, H, W] squared error per token
    r2 = r.pow(2).sum(-1)
    if bulk is None:
        bulk = torch.ones_like(e2, dtype=torch.bool)
    bulk = bulk.cpu()
    bulk_err = float(e2[bulk].sum().sqrt() / r2[bulk].sum().sqrt().clamp_min(1e-30))
    rms = r2.mean(dim=(1, 2), keepdim=True).sqrt().clamp_min(1e-30)
    tok = torch.where(bulk, e2.sqrt() / rms, torch.zeros_like(e2))
    at = np.unravel_index(int(tok.argmax()), tuple(tok.shape))
    regs, ratio = {}, 0.0
    for name, m in regions.items():
        m = m.cpu()
        n = int(m.sum())
        if n == 0:
            continue
        err = float(e2[m].sum().sqrt() / r2[m].sum().sqrt().clamp_min(1e-30))
        regs[name] = (err, n)
        if n >= MIN_REGION:
            ratio = max(ratio, err / max(bulk_err, 1e-30))
    return {"bulk": bulk_err, "regions": regs, "token": float(tok.max()), "token_at": tuple(int(v) for v in at),
            "ratio": ratio}


def check_regions(rep: dict, what: str, ratio: float = 3.0, token_ratio: float = 10.0) -> None:
    """Every region of at least MIN_REGION tokens within ``ratio`` x the bulk error, every bulk token within
    ``token_ratio`` x the bulk error; a failure names the worst regions."""
    bulk = rep["bulk"]
    worst = sorted(((e / max(bulk, 1e-30), name, e, n) for name, (e, n) in rep["regions"].items() if n >= MIN_REGION),
                   reverse=True)
    where = ", ".join(f"{name} {e:.2e} ({q:.1f}x, {n} tokens)" for q, name, e, n in worst[:5])
    assert not worst or worst[0][0] <= ratio, f"{what}: bulk rel-L2 {bulk:.2e}; worst regions: {where}"
    assert rep["token"] <= token_ratio * bulk, \
        f"{what}: token {rep['token_at']} off by {rep['token']:.2e} of the frame's RMS token norm (bulk {bulk:.2e}); {where}"


def ref_keys():
    with open(os.path.join(GOLDEN, "state_dict_keys.json")) as fh:
        return json.load(fh)


class FusionCase:
    """One golden fusion fixture + everything needed to re-run it."""

    def __init__(self, tag):
        z = np.load(os.path.join(GOLDEN, f"fusion_{tag}.npz"))
        self.tag, self.z = tag, z
        geometry, level, batch, layers, chg, nsk = [str(v) for v in z["meta"]]
        self.geometry, self.level, self.batch = geometry, int(level), int(batch)
        self.layers = tuple(layers.split(","))
        self.change_embedding, self.no_skip_inside = bool(int(chg)), bool(int(nsk))
        self.C, _, self.max_res, self.large_kernel = synth.LEVELS[self.level]
        self.geo = dict(zip([str(k) for k in z["geo_keys"]], [int(v) for v in z["geo_vals"]]))
        self.offsets = (self.geo["offset_y"], self.geo["offset_x"])
        kind = "baseline" if self.layers == synth.BASELINE_LAYERS else "combine1"
        self.shapes = ref_keys()[f"fusion_{kind}_L{self.level}"]
        self.hist_shapes = ref_keys()["hist_encoder"]

    def inputs(self):
        return synth.make_inputs(self.geometry, self.batch, seed=1, levels=(self.level,))

    def state_dict(self):
        return synth.synthetic_state_dict(self.shapes, seed=self.level)

    def hist_state_dict(self):
        return synth.synthetic_state_dict(self.hist_shapes, seed=0)

    def mask_bits(self, name):
        shape = tuple(int(v) for v in self.z[f"{name}_shape"])
        n = int(np.prod(shape))
        return np.unpackbits(self.z[f"{name}_bits"])[:n].reshape(shape).astype(bool)

    def check_output(self, out: torch.Tensor, tol: float, what: str):
        """out [B,C,H,W] vs the stored reference output (full or sampled)."""
        out = out.detach().double().cpu()
        z = self.z
        assert tuple(out.shape) == tuple(int(v) for v in z["out_shape"]), what
        assert torch.isfinite(out).all(), what
        if "out_full" in z.files:
            err = rel_l2(out, torch.from_numpy(z["out_full"]))
            assert err <= tol, f"{what}: rel-L2 {err:.3e} > {tol:.1e}"
            return err
        idx = torch.from_numpy(z["out_idx"])
        e1 = rel_l2(out.reshape(-1)[idx], torch.from_numpy(z["out_sample"]))
        e2 = rel_l2(out.sum(dim=1), torch.from_numpy(z["out_chansum"]))
        e3 = rel_l2(out.sum(dim=(2, 3)), torch.from_numpy(z["out_perchan"]))
        # sums over C (or H*W) elements shrink relative errors of independent noise but keep
        # systematic ones; same tolerance on all three
        assert e1 <= tol and e2 <= tol and e3 <= tol, \
            f"{what}: rel-L2 sample {e1:.3e} chansum {e2:.3e} perchan {e3:.3e} > {tol:.1e}"
        return max(e1, e2, e3)
