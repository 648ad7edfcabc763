"""The tail_b16 workload (bench.py --workload tail_b16: histogram encoder + Decoder with its three fusion calls + DepthHead,
16 frames at 416x544, the same seeded weights and inputs) on both engines of the decoder shell and head, alternating in
one process: the exact fp32 engine (Decoder.compute_dtype = torch.float32, fusion modules in fp32) and the bf16 tensor-core
engine.  Prints one JSON line per engine and round: step time from CUDA events, frames/s, the card's name and power limit
read in the same run, and the algorithmic GFLOP/frame.

    python tools/tail_f32_bench.py [--steps 10] [--warmup 3] [--rounds 1]
"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import cfpnet_b200  # noqa: E402
from cfpnet_b200 import decoder as D, shard, synth  # noqa: E402
from cfpnet_b200.build import build  # noqa: E402
from cfpnet_b200.config import args as cargs  # noqa: E402

GEOMETRY = "G416"
FUSION_FLOP_PER_FRAME = 13.22e9           # the three fusion calls at 416x544 (bench.py FLOP_PER_FRAME)


def decoder_head_flop_per_frame(img_h, img_w):
    """Useful flops of the decoder shell's convs (decoder.py:70-80, 43-48), DepthRegression.conv3x3 and conv_out for one
    frame: 2 x pixels x cin x cout x taps each (38.4 GFLOP at 416x544)."""
    px = {s: (img_h // s) * (img_w // s) for s in (2, 4, 8, 16, 32)}
    convs = [(px[32], 232, 256, 1), (px[16], 392, 256, 9), (px[16], 256, 256, 9), (px[16], 256, 128, 1),
             (px[8], 312, 128, 9), (px[8], 128, 128, 9), (px[8], 128, 64, 1),
             (px[4], 168, 64, 9), (px[4], 64, 64, 9), (px[4], 64, 32, 1),
             (px[2], 80, 32, 9), (px[2], 32, 32, 9), (px[2], 32, 128, 9), (px[2], 128, 128, 9),
             (px[2], 128, 256, 1)]
    return sum(2.0 * p * ci * co * t for p, ci, co, t in convs)


def gpu_identity():
    """(name, power limit in W or None) of cuda:0, read now."""
    props = torch.cuda.get_device_properties(0)
    limit = None
    for sel in (f"GPU-{props.uuid}", "0"):
        try:
            r = subprocess.run(["nvidia-smi", f"--id={sel}", "--query-gpu=power.limit", "--format=csv,noheader,nounits"],
                               capture_output=True, text=True, timeout=30)
            if r.returncode == 0 and r.stdout.strip():
                limit = float(r.stdout.strip().splitlines()[0])
                break
        except (OSError, ValueError, subprocess.TimeoutExpired):
            pass
    return props.name, limit


def make_engine(sd, dev, dtype):
    dec = D.Decoder(num_classes=128)
    dec.load_state_dict({k[len("decoder."):]: v for k, v in sd.items() if k.startswith("decoder.")}, strict=True)
    dec = dec.to(dev).eval()
    dec.compute_dtype = dtype
    if dtype == torch.bfloat16:
        for m in (dec.cross_atten1, dec.cross_atten2, dec.cross_atten3):
            m.to(torch.bfloat16)
    enc = cfpnet_b200.HistogramEncoder()
    enc.load_state_dict({k[len("hist_encoder."):]: v for k, v in sd.items() if k.startswith("hist_encoder.")}, strict=True)
    enc = enc.to(dev).eval()
    enc.out_dtype = dtype
    head = D.DepthHead(n_bins=256, min_val=1e-3, max_val=10.0)
    head.load_state_dict({k: v for k, v in sd.items() if k.startswith(("depth_head.", "conv_out."))}, strict=True)
    return enc, dec, head.to(dev).eval()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=1, help="fp32 / bf16 measurement pairs, alternating")
    ap.add_argument("--batch", type=int, default=16)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("tail_f32_bench.py needs a CUDA device: the path has no CPU fallback")
    torch.cuda.set_device(0)
    dev = torch.device("cuda", 0)
    build()
    B = a.batch
    cargs.attention_layer = list(synth.COMBINE1_LAYERS)
    with open(os.path.join(ROOT, "tests", "golden", "depth_tail_keys.json")) as fh:
        sd = synth.synthetic_state_dict(json.load(fh), seed=11)
    engines = {"fp32": make_engine(sd, dev, torch.float32), "bf16": make_engine(sd, dev, torch.bfloat16)}
    sets = []
    for s_ in range(3):
        inp = synth.make_inputs(GEOMETRY, B, seed=200 + s_, levels=())
        d = {f"f{i}": t.to(dev) for i, t in enumerate(synth.encoder_features(GEOMETRY, B, seed=200 + s_))}
        d["hist_data"], d["mask"] = inp["hist_data"].to(dev), inp["mask"].to(dev)
        sets.append(d)
    patch_info = inp["patch_info"]
    img_h, img_w, _ = synth.GEOMETRIES[GEOMETRY]
    dec_flop = decoder_head_flop_per_frame(img_h, img_w)

    def step(name, d, i):
        enc, dec, head = engines[name]
        shard.seed_posenc(i)
        hist = enc(d["hist_data"].unsqueeze(-1))
        unet, H, W = dec.forward_nhwc([d[f"f{j}"] for j in range(5)], hist, rect_data=None, mask=d["mask"], patch_info=patch_info, rgb=None)
        return head.forward_nhwc(unet, H, W)

    with torch.no_grad():
        for r in range(a.rounds):
            for name in ("fp32", "bf16"):
                for i in range(max(a.warmup, 1)):
                    step(name, sets[i % 3], i)
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for i in range(a.steps):
                    step(name, sets[i % 3], i)
                e1.record()
                torch.cuda.synchronize()
                ms = e0.elapsed_time(e1) / a.steps
                gpu, limit = gpu_identity()
                print(json.dumps({
                    "workload": f"tail_b{B}", "engine": name, "round": r, "batch": B, "image": [img_h, img_w], "steps": a.steps,
                    "warmup": max(a.warmup, 1), "ms_per_step": ms, "frames_per_s": B / (ms * 1e-3),
                    "decoder_head_gflop_per_frame": dec_flop / 1e9, "fusion_gflop_per_frame": FUSION_FLOP_PER_FRAME / 1e9,
                    "decoder_head_fusion_tflops": B * (dec_flop + FUSION_FLOP_PER_FRAME) / (ms * 1e-3) / 1e12,
                    "gpu": gpu, "power_limit_w": limit}), flush=True)


if __name__ == "__main__":
    main()
