"""Batch-1 latency of the model below the image encoder (histogram encoder -> Decoder with its three fusion calls -> DepthHead)
on both engines, eager and as one CUDA-graph replay (cfpnet_b200.pipeline.make_graphed_depth), with the reference's
evaluate_time.py protocol: 100 warm-up forwards, then 500 forwards each bracketed by torch.cuda.synchronize(), reported as the
trimmed mean sum(sorted(dt)[1:-2]) / 497.  Same seeded weights as tools/tail_f32_bench.py (depth_tail_keys.json, seed 11).

Workloads: G480 (480x640, 8x8 zones of 56 px, 256 bins; L3 takes hist2image's resize branch, every map fills its positional-
encoding table) and G416 (416x544, 48 px zones; six crop draws per forward), B = 1.  Eager / graph and fp32 / bf16 alternate
within one process: both orders flip on odd rounds.  One JSON line per (geometry, engine, mode, round): ms, median, min,
libcfp launches per eager forward, the host cost of the graph's staleness check, the card's name and power limit read in the
same run.  A
separate pass then takes the per-kernel time shares of one eager forward from cfp_profile_start / cfp_profile_stop
(mode "kernel_split").

    python tools/depth_latency_bench.py [--rounds 2] [--warmup 100] [--iters 500]
"""
import argparse
import json
import os
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from cfpnet_b200 import _lib, shard, synth  # noqa: E402
from cfpnet_b200.build import build  # noqa: E402
from cfpnet_b200.config import args as cargs  # noqa: E402
from cfpnet_b200.pipeline import make_graphed_depth  # noqa: E402
from tail_f32_bench import gpu_identity, make_engine  # noqa: E402

GEOMETRIES = ("G480", "G416")
ENGINES = {"fp32": torch.float32, "bf16": torch.bfloat16}


def eager_forward(model, d):
    enc, dec, head = model
    hist = enc(d["hist_data"].unsqueeze(-1))
    unet, H, W = dec.forward_nhwc(d["feats"], hist, rect_data=None, mask=d["mask"], patch_info=d["patch_info"], rgb=None)
    return head.forward_nhwc(unet, H, W)


def time_forwards(fn, warmup, iters):
    """evaluate_time.py: warm-up, then per-forward host time between two device synchronisations."""
    for i in range(warmup):
        shard.seed_posenc(i)
        fn()
    torch.cuda.synchronize()
    dt = []
    for i in range(iters):
        shard.seed_posenc(i)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        dt.append(time.perf_counter() - t0)
    s = sorted(dt)
    trimmed = s[1:-2] if len(s) > 3 else s
    return 1e3 * sum(trimmed) / len(trimmed), 1e3 * s[len(s) // 2], 1e3 * s[0]


def guard_us(run, n=2000):
    run.check()
    t0 = time.perf_counter()
    for _ in range(n):
        run.check()
    return 1e6 * (time.perf_counter() - t0) / n


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=2, help="eager / graph x fp32 / bf16 measurement sets, alternating")
    ap.add_argument("--warmup", type=int, default=100)
    ap.add_argument("--iters", type=int, default=500)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("depth_latency_bench.py needs a CUDA device: the path has no CPU fallback")
    torch.cuda.set_device(0)
    dev = torch.device("cuda", 0)
    build()
    cargs.attention_layer = list(synth.COMBINE1_LAYERS)
    with open(os.path.join(ROOT, "tests", "golden", "depth_tail_keys.json")) as fh:
        sd = synth.synthetic_state_dict(json.load(fh), seed=11)
    models = {name: make_engine(sd, dev, dt) for name, dt in ENGINES.items()}
    data = {}
    for geo in GEOMETRIES:
        inp = synth.make_inputs(geo, 1, seed=200, levels=())
        data[geo] = dict(feats=[t.to(dev) for t in synth.encoder_features(geo, 1, seed=200)], hist_data=inp["hist_data"].to(dev),
                         mask=inp["mask"].to(dev), patch_info=inp["patch_info"])
    img = {geo: list(synth.GEOMETRIES[geo][:2]) for geo in GEOMETRIES}

    with torch.no_grad():
        launches, graphs = {}, {}
        for geo in GEOMETRIES:
            d = data[geo]
            for name, model in models.items():
                eager_forward(model, d)                       # packs the weights, sizes the scratch
                torch.cuda.synchronize()
                n0 = _lib.launch_count()
                eager_forward(model, d)
                launches[geo, name] = _lib.launch_count() - n0
                graphs[geo, name] = make_graphed_depth(*model, d["feats"], d["hist_data"], d["mask"], d["patch_info"])
        for r in range(a.rounds):
            for geo in GEOMETRIES:
                d = data[geo]
                engines = list(models.items())
                for name, model in (engines if r % 2 == 0 else engines[::-1]):
                    run = graphs[geo, name]
                    modes = (("eager", lambda: eager_forward(model, d)),
                             ("graph", lambda: run(d["feats"], d["hist_data"], d["mask"])))
                    for mode, fn in (modes if r % 2 == 0 else modes[::-1]):
                        ms, med, mn = time_forwards(fn, a.warmup, a.iters)
                        gpu, limit = gpu_identity()
                        print(json.dumps({
                            "workload": f"depth_latency_{geo}", "geometry": geo, "image": img[geo], "batch": 1, "engine": name,
                            "mode": mode, "round": r, "warmup": a.warmup, "iters": a.iters, "ms": ms, "median_ms": med, "min_ms": mn,
                            "cfp_launch_count_per_eager_forward": launches[geo, name], "guard_check_us": guard_us(run),
                            "gpu": gpu, "power_limit_w": limit}), flush=True)
        # kernel split: events around every libcfp launch of one eager forward (profiling slows the host: not timed above)
        for geo in GEOMETRIES:
            for name, model in models.items():
                shard.seed_posenc(0)
                eager_forward(model, data[geo])
                torch.cuda.synchronize()
                _lib.profile_start()
                shard.seed_posenc(0)
                eager_forward(model, data[geo])
                torch.cuda.synchronize()
                prof = _lib.profile_stop()
                total = sum(v[1] for v in prof.values())
                split = sorted(((k, n, t) for k, (n, t) in prof.items()), key=lambda x: -x[2])
                gpu, limit = gpu_identity()
                print(json.dumps({
                    "workload": f"depth_latency_{geo}", "geometry": geo, "image": img[geo], "batch": 1, "engine": name,
                    "mode": "kernel_split", "kernel_ms_total": total,
                    "kernels": [{"kernel": k, "launches": n, "ms": t, "share": t / total if total else None} for k, n, t in split],
                    "gpu": gpu, "power_limit_w": limit}), flush=True)


if __name__ == "__main__":
    main()
