"""One training step of the whole model below the image encoder on libcfp, 16 frames at 416x544 with seeded weights and
inputs: zero_grad -> histogram encoder -> Decoder (three fusion calls) -> DepthHead, all in .train() -> SILogLoss against a
seeded target -> backward -> FlatTrainer update (clip + AdamW).  Prints one JSON line per round: ms per step from CUDA
events, frames/s, libcfp launches per step, peak device memory, and the card's name and power limit read in the same run.
``--profile`` adds one torch.profiler run (separate from the timed rounds) and prints the GPU-time share of the conv
weight gradient, the conv input gradient and the forward convs.

    python tools/train_tail_bench.py [--steps 5] [--warmup 2] [--rounds 2] [--profile]
"""
import argparse
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import cfpnet_b200  # noqa: E402
from cfpnet_b200 import _lib, decoder as D, shard, synth  # noqa: E402
from cfpnet_b200.build import build  # noqa: E402
from cfpnet_b200.config import args as cargs  # noqa: E402
from cfpnet_b200.loss import SILogLoss  # noqa: E402
from cfpnet_b200.train import FlatTrainer  # noqa: E402
from tail_f32_bench import FUSION_FLOP_PER_FRAME, decoder_head_flop_per_frame, gpu_identity  # noqa: E402

GEOMETRY = "G416"


def make_model(sd, dev):
    enc = cfpnet_b200.HistogramEncoder()
    enc.load_state_dict({k[len("hist_encoder."):]: v for k, v in sd.items() if k.startswith("hist_encoder.")}, strict=True)
    dec = D.Decoder(num_classes=128)
    dec.load_state_dict({k[len("decoder."):]: v for k, v in sd.items() if k.startswith("decoder.")}, strict=True)
    head = D.DepthHead(n_bins=256, min_val=1e-3, max_val=10.0)
    head.load_state_dict({k: v for k, v in sd.items() if k.startswith(("depth_head.", "conv_out."))}, strict=True)
    return enc.to(dev).train(), dec.to(dev).train(), head.to(dev).train()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--batch", type=int, default=16)
    ap.add_argument("--profile", action="store_true", help="one extra torch.profiler step: time share of wgrad / dgrad / forward convs")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("train_tail_bench.py needs a CUDA device: the path has no CPU fallback")
    torch.cuda.set_device(0)
    dev = torch.device("cuda", 0)
    build()
    B = a.batch
    cargs.attention_layer = list(synth.COMBINE1_LAYERS)
    with open(os.path.join(ROOT, "tests", "golden", "depth_tail_keys.json")) as fh:
        sd = synth.synthetic_state_dict(json.load(fh), seed=11)
    enc, dec, head = make_model(sd, dev)
    trainer = FlatTrainer([enc, dec, head], lr=1e-4)
    loss_fn = SILogLoss()
    img_h, img_w, _ = synth.GEOMETRIES[GEOMETRY]
    sets = []
    for s_ in range(2):
        inp = synth.make_inputs(GEOMETRY, B, seed=300 + s_, levels=())
        d = {f"f{i}": t.to(dev) for i, t in enumerate(synth.encoder_features(GEOMETRY, B, seed=300 + s_))}
        d["hist_data"], d["mask"] = inp["hist_data"].to(dev), inp["mask"].to(dev)
        d["target"] = (torch.rand(B, 1, img_h, img_w, generator=torch.Generator().manual_seed(400 + s_)) * 4 + 0.5).to(dev)
        sets.append(d)
    patch_info = inp["patch_info"]
    dec_flop = decoder_head_flop_per_frame(img_h, img_w)

    def step(d, i):
        trainer.zero_grad()
        shard.seed_posenc(i)
        hist = enc(d["hist_data"].unsqueeze(-1))
        unet = dec([d[f"f{j}"] for j in range(5)], hist, rect_data=None, mask=d["mask"], patch_info=patch_info, rgb=None)
        _, pred = head(unet)
        loss = loss_fn(pred, d["target"])
        loss.backward()
        trainer.update()
        return loss

    for i in range(max(a.warmup, 1)):
        step(sets[i % 2], i)
    torch.cuda.synchronize()
    for r in range(a.rounds):
        torch.cuda.reset_peak_memory_stats(dev)
        n0 = _lib.launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(a.steps):
            loss = step(sets[i % 2], i)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / a.steps
        gpu, limit = gpu_identity()
        print(json.dumps({
            "workload": f"train_tail_b{B}", "round": r, "batch": B, "image": [img_h, img_w], "steps": a.steps,
            "warmup": max(a.warmup, 1), "ms_per_step": ms, "frames_per_s": B / (ms * 1e-3),
            "libcfp_launches_per_step": (_lib.launch_count() - n0) / a.steps,
            "peak_mem_gb": torch.cuda.max_memory_allocated(dev) / 1e9, "loss": float(loss),
            "decoder_head_gflop_per_frame_fwd": dec_flop / 1e9, "fusion_gflop_per_frame_fwd": FUSION_FLOP_PER_FRAME / 1e9,
            "gpu": gpu, "power_limit_w": limit}), flush=True)

    if a.profile:
        def kernel_us(fn):
            with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
                fn()
                torch.cuda.synchronize()
            out = {"total": 0.0, "wgrad": 0.0, "conv_f32": 0.0}
            for e in prof.key_averages():
                t = getattr(e, "device_time_total", 0.0)
                out["total"] += t
                if "conv_wgrad" in e.key or "sum_partials" in e.key:
                    out["wgrad"] += t
                elif "conv_f32_kernel" in e.key:
                    out["conv_f32"] += t
            return out

        def forward_only():
            with torch.no_grad():
                hist = enc(sets[0]["hist_data"].unsqueeze(-1))
                head(dec([sets[0][f"f{j}"] for j in range(5)], hist, rect_data=None, mask=sets[0]["mask"], patch_info=patch_info,
                         rgb=None))

        # forward convs and input gradients run the same kernel: the forward's share comes from a forward-only pass
        whole, fwd = kernel_us(lambda: step(sets[0], 0)), kernel_us(forward_only)
        tot = max(whole["total"], 1e-9)
        print(json.dumps({"profile": f"train_tail_b{B} step (torch.profiler, separate run)", "gpu_ms": whole["total"] / 1e3,
                          "share_conv_wgrad": whole["wgrad"] / tot, "share_conv_forward": fwd["conv_f32"] / tot,
                          "share_conv_dgrad": (whole["conv_f32"] - fwd["conv_f32"]) / tot}), flush=True)


if __name__ == "__main__":
    main()
