"""helpers.region_errors / check_regions without a GPU: a map with bf16-level noise everywhere (rel-L2 ~9e-3, what the
bf16 engine measures) and one local defect of 5-10 % of the signal.  Each defect passes the whole-map bound the bf16
parity tests use (2e-2) and fails the per-region check - the blind spot of a global rel-L2, in numbers."""
import pytest
import torch

from helpers import check_regions, region_errors, rel_l2

B, H, W, C, K = 32, 30, 40, 32, 7          # the L3 map of a 480x640 image, 32 frames, k = 7: bands of (K - 1) / 2 = 3 cells
P = (K - 1) // 2
GLOBAL_BF16 = 2e-2                         # tests/test_gpu_parity.py::BF16_TOL


def regions():
    """The regions the GPU sweeps check: frames, raster 128-token tiles over the whole batch, per-frame border bands, and
    columns (a column-indexing error hits every frame)."""
    regs = {}
    for b in range(B):
        m = torch.zeros(B, H, W, dtype=torch.bool)
        m[b] = True
        regs[f"frame {b}"] = m
        for side, sl in (("top", (slice(0, P), slice(None))), ("bottom", (slice(H - P, H), slice(None))),
                         ("left", (slice(None), slice(0, P))), ("right", (slice(None), slice(W - P, W)))):
            m = torch.zeros(B, H, W, dtype=torch.bool)
            m[b][sl] = True
            regs[f"frame {b} {side} band"] = m
    flat = torch.arange(B * H * W).reshape(B, H, W)
    for t in range((B * H * W + 127) // 128):
        regs[f"tile {t}"] = (flat // 128) == t
    for x in range(W):
        m = torch.zeros(B, H, W, dtype=torch.bool)
        m[:, :, x] = True
        regs[f"column {x}"] = m
    return regs


REGIONS = regions()


def noisy_pair(seed):
    g = torch.Generator().manual_seed(seed)
    ref = torch.randn(B, H, W, C, generator=g, dtype=torch.float64)
    out = ref + 9e-3 * torch.randn(B, H, W, C, generator=g, dtype=torch.float64)
    return out, ref


def test_noise_alone_passes_both_checks():
    out, ref = noisy_pair(0)
    assert rel_l2(out, ref) <= GLOBAL_BF16
    rep = region_errors(out, ref, REGIONS)
    assert 8e-3 <= rep["bulk"] <= 1e-2
    check_regions(rep, "bf16-level noise")


def defect(name):
    """Token mask of the defect and its relative size (5 - 10 %)."""
    m = torch.zeros(B, H, W, dtype=torch.bool)
    if name == "tile":
        m.view(-1)[128 * 77:128 * 78] = True                        # one 128-token tile, straddling frames 8 and 9
        amp = 0.10
    elif name == "column":
        m[:, :, 17] = True                                          # one image column, every frame
        amp = 0.07
    elif name == "last frame of a stack":
        m[2] = True                                                 # frames stacked 3 to a plane: the third of the first stack
        amp = 0.07
    elif name == "border band":
        m[5, :, W - P:] = True                                      # the right halo band of one frame
        amp = 0.10
    return m, amp


@pytest.mark.parametrize("name", ["tile", "column", "last frame of a stack", "border band"])
def test_local_defect_passes_the_global_bound_and_fails_the_region_check(name):
    out, ref = noisy_pair(1)
    g = torch.Generator().manual_seed(2)
    m, amp = defect(name)
    # a systematic error of `amp` of the signal on the defect's tokens (a wrong tap, a wrong row, a stale operand ...)
    out = torch.where(m[..., None], out + amp * torch.randn(B, H, W, C, generator=g, dtype=torch.float64).mul(ref.abs()), out)
    err = rel_l2(out, ref)
    assert err <= GLOBAL_BF16, f"{name}: the defect should hide under the global bound, rel-L2 {err:.3e}"
    rep = region_errors(out, ref, REGIONS)
    with pytest.raises(AssertionError) as exc:
        check_regions(rep, name)
    # the report names the worst region first, and that region overlaps the defect
    worst = max((e, k) for k, (e, n) in rep["regions"].items() if n >= 16)[1]
    assert REGIONS[worst][m].any(), worst
    assert f"worst regions: {worst} " in str(exc.value), str(exc.value)


def test_bulk_excludes_tokens_the_layer_leaves_alone():
    """With a bulk mask, tokens outside it count neither in the bulk error nor in the per-token figure."""
    out, ref = noisy_pair(3)
    bulk = torch.zeros(B, H, W, dtype=torch.bool)
    bulk[:, 5:20, 10:30] = True
    out = torch.where(bulk[..., None], out, ref)                     # exact outside the bulk
    rep = region_errors(out, ref, {"outside": ~bulk}, bulk=bulk)
    assert 8e-3 <= rep["bulk"] <= 1e-2
    assert rep["regions"]["outside"][0] == 0.0
    assert rep["token_at"][1] in range(5, 20) and rep["token_at"][2] in range(10, 30)
