"""The fusion path as one callable: histogram encoder + the three ``TransformerFusion``
calls of the reference decoder (``cross_atten3`` at 1/16, ``cross_atten2`` at 1/8,
``cross_atten1`` at 1/4; ``src/models/decoder.py:90-94,111,116,121``, ``deltar.py:40``).

One *frame* of BASELINE.json's metric is exactly this work for one image.  The
class only wires the drop-in modules together the way ``Deltar`` / ``Decoder`` do and
adds the host<->device staging used for the end-to-end measurement.
"""
from __future__ import annotations

from typing import Dict, Iterable, Iterator, List, Sequence, Tuple

import torch
import torch.nn as nn

from .config import args
from .encoder import HistogramEncoder
from .fusion import TransformerFusion
from .synth import LEVELS


class FusionPath(nn.Module):
    def __init__(self, layer_names: Sequence[str] | None = None):
        super().__init__()
        if layer_names is not None:
            args.attention_layer = list(layer_names)
        self.hist_encoder = HistogramEncoder()
        # same constructor arguments as decoder.py:92-94
        self.cross_atten1 = TransformerFusion(embedding_dim=32, max_resolution=[120, 160], large_kernel=31, patch_size=16)
        self.cross_atten2 = TransformerFusion(embedding_dim=64, max_resolution=[60, 80], large_kernel=15, patch_size=8)
        self.cross_atten3 = TransformerFusion(embedding_dim=128, max_resolution=[30, 40], large_kernel=7, patch_size=4)
        self._pinned_out = None

    def set_dtype(self, dtype: torch.dtype) -> "FusionPath":
        self.to(dtype)
        self.hist_encoder.out_dtype = dtype
        return self

    # run the three fusion calls of the synthetic harness on three streams (CFP_SEQUENTIAL_LEVELS=1: one stream, the drop-in order)
    concurrent_levels = not bool(__import__("os").environ.get("CFP_SEQUENTIAL_LEVELS"))

    def forward(self, x3, x2, x1, hist_data, mask, patch_info, rect_data=None, ready=None, done=None) -> List[torch.Tensor]:
        """x3/x2/x1: decoder features [B,128,h/16,w/16], [B,64,h/8,w/8], [B,32,h/4,w/4];
        hist_data [B,Z,S]; mask [B,Z] bool.  Returns the fused maps in call order.

        In THIS harness the three level inputs are given up front (synthetic decoder features), so the three
        TransformerFusion calls are independent and are enqueued on three streams: their (mostly latency-bound) kernels
        overlap on the GPU.  Inside the reference's ``Decoder`` they are NOT independent - ``x_d2`` is computed from the
        fused ``x_d3`` and ``x_d1`` from the fused ``x_d2`` (``decoder.py:109-121``) - so a drop-in there runs them one
        after the other: ``concurrent_levels = False`` (or ``CFP_SEQUENTIAL_LEVELS=1``) is that configuration, and
        ``bench.py`` reports it next to the headline as ``drop_in_sequential``; ``cfpnet_b200.decoder.Decoder`` is the
        integrated form.  The host-side order of the calls - and with it the order of the positional-encoding RNG
        draws - stays L3, L2, L1 as in the reference decoder.

        ``ready`` / ``done`` (used by :meth:`stream_host`): CUDA events per input - ``ready["hist"]`` (histograms and mask),
        ``ready["x3"]``, ``["x2"]``, ``["x1"]`` - that the consuming stream waits for right before its first use, and one
        event per level, recorded when that level's fused map is complete.  With them a level starts as soon as ITS inputs have
        landed and its result can leave as soon as it exists, instead of the whole call waiting for the largest map either way.
        Created with ``external=True`` they stay external wait / record nodes when the call is captured into a CUDA graph."""
        if ready is not None and x3.is_cuda:
            torch.cuda.current_stream(x3.device).wait_event(ready["hist"])
        f32, f64, f128 = self.hist_encoder(hist_data.unsqueeze(-1))
        kw = dict(rect_data=rect_data, mask=mask, patch_info=patch_info, rgb=None)
        jobs = ((self.cross_atten3, x3, f128), (self.cross_atten2, x2, f64), (self.cross_atten1, x1, f32))
        names = ("x3", "x2", "x1")
        if not (self.concurrent_levels and x3.is_cuda):
            outs = []
            for i, (m, x, f) in enumerate(jobs):
                if ready is not None and x.is_cuda:
                    torch.cuda.current_stream(x.device).wait_event(ready[names[i]])
                outs.append(m(x, f, **kw))
                if done is not None and x.is_cuda:
                    done[i].record(torch.cuda.current_stream(x.device))
            return outs
        dev = x3.device
        cur = torch.cuda.current_stream(dev)
        # (measured: stream priorities do not help - higher priority for the two smaller levels costs 2.5 %, for the
        # largest level nothing changes)
        side = self.__dict__.setdefault("_level_streams", {}).setdefault(str(dev), [torch.cuda.Stream(dev) for _ in range(2)])
        # results are allocated on the caller's stream (no cross-stream allocator traffic: record_stream()
        # on side-stream tensors turns into a cudaMalloc per step, and those occasionally stall for ~100 ms)
        outs = [torch.empty_like(x, memory_format=torch.contiguous_format) for _, x, _ in jobs]
        fork = torch.cuda.Event()
        fork.record(cur)
        joins = []
        # programmatic dependent launch pays on one stream; with three streams the pre-launched CTAs only take slots
        # from the other levels' kernels (measured: -3.5 % sequential, +1.5 % concurrent) - off for this region
        from . import _lib
        prev_pdl = _lib.set_pdl(False)
        try:
            for i, (m, x, f) in enumerate(jobs):
                if i == 2:                                   # the largest level stays on the caller's stream
                    if ready is not None:
                        cur.wait_event(ready[names[i]])
                    m(x, f, out=outs[i], **kw)
                    if done is not None:
                        done[i].record(cur)
                    continue
                s = side[i]
                s.wait_event(fork)
                if ready is not None:
                    s.wait_event(ready[names[i]])
                with torch.cuda.stream(s):
                    m(x, f, out=outs[i], **kw)
                    if done is not None:
                        done[i].record(s)
                    e = torch.cuda.Event()
                    e.record(s)
                joins.append(e)
        finally:
            _lib.set_pdl(bool(prev_pdl))
        for e in joins:
            cur.wait_event(e)
        return outs

    # ------------------------------------------------------------------ CUDA-graph replay (latency mode)
    def make_graphed(self, x3, x2, x1, hist_data, mask, patch_info, copy_inputs: bool = True, ready=None, done=None):
        """Capture one forward (every launch of the three levels, on all their streams) into a CUDA graph and return
        ``run(x3, x2, x1, hist_data, mask) -> [fused3, fused2, fused1]`` that replays it: the ~95 host-side launches of
        a forward (~20 us each through Python + ctypes) become one graph launch.  ``copy_inputs``: the arguments of
        ``run`` are copied into the captured static buffers first; with ``copy_inputs=False`` the captured tensors ARE the
        inputs (``run()`` takes no arguments; the caller refills them in place).

        The positional-encoding crop offsets (``fusion.py:88-91``, drawn per forward when a map is smaller than its
        table) are not frozen into the graph: while capturing, the modules read them from a small device buffer
        (``cfp_posenc_tokens_crop_fwd``), and every replay first makes the reference's draws - same generator, same
        order L3, L2, L1 - and uploads them."""
        mods = ((self.cross_atten3, x3), (self.cross_atten2, x2), (self.cross_atten1, x1))
        static = [t.clone() for t in (x3, x2, x1, hist_data, mask)] if copy_inputs else [x3, x2, x1, hist_data, mask]
        dev = x3.device
        crop_dev = torch.zeros(3, 2, device=dev, dtype=torch.int32)
        shapes = [(m, int(x.shape[2]), int(x.shape[3])) for m, x in mods]

        def upload_crops():
            vals = [list(m.draw_crop(H, W)) for m, H, W in shapes]
            crop_dev.copy_(torch.tensor(vals, dtype=torch.int32))       # stream-ordered before the replay

        side = torch.cuda.Stream(dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        try:
            for i, (m, _x) in enumerate(mods):
                m.__dict__["_crop_dev"] = crop_dev[i]
            with torch.cuda.stream(side), torch.no_grad():          # warm-up off the capture: packing, scratch, smem attributes
                for _ in range(2):
                    self.forward(*static, patch_info)
            torch.cuda.current_stream(dev).wait_stream(side)
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph), torch.no_grad():   # ready / done: external wait / record nodes of the graph
                outs = self.forward(*static, patch_info, ready=ready, done=done)
        finally:
            for m, _x in mods:
                m.__dict__.pop("_crop_dev", None)

        def run(*inputs):
            if copy_inputs:
                for dst, src in zip(static, inputs):
                    dst.copy_(src, non_blocking=True)
            upload_crops()
            graph.replay()
            return outs

        run.graph, run.crop_dev, run.static = graph, crop_dev, static
        return run

    # ------------------------------------------------------------------ host-buffer entry
    def forward_host(self, host: Dict[str, torch.Tensor], patch_info, device) -> List[torch.Tensor]:
        """End-to-end call with HOST buffers: pinned inputs are copied to the device, the path
        runs, and the three fused maps are read back into pinned host memory."""
        dev = {k: host[k].to(device, non_blocking=True) for k in ("x3", "x2", "x1", "hist_data", "mask")}
        outs = self.forward(dev["x3"], dev["x2"], dev["x1"], dev["hist_data"], dev["mask"], patch_info)
        if self._pinned_out is None or any(p.shape != o.shape or p.dtype != o.dtype
                                           for p, o in zip(self._pinned_out, outs)):
            self._pinned_out = [torch.empty(o.shape, dtype=o.dtype, pin_memory=True) for o in outs]
        for p, o in zip(self._pinned_out, outs):
            p.copy_(o, non_blocking=True)
        torch.cuda.current_stream(device).synchronize()
        return self._pinned_out

    # ------------------------------------------------------------------ pipelined host-buffer entry
    def stream_host(self, batches: Iterable[Dict[str, torch.Tensor]], patch_info, device, depth: int = 3,
                    seeds: Iterable[int] | None = None, graph: bool = False) -> Iterator[Tuple[int, List[torch.Tensor]]]:
        """Throughput form of :meth:`forward_host`: yields ``(index, [fused3, fused2, fused1])`` (pinned host
        tensors, valid until ``depth`` more batches have been yielded) for every batch of pinned host inputs.

        Three streams overlap the stages of consecutive batches: host->device copies of batch i+1 run
        on a copy stream while batch i computes and the results of batch i-1 travel back on a third
        stream.  Every batch still pays its full H2D + D2H; nothing is cached across batches.
        ``seeds`` (one int per batch) seeds the positional-encoding crop before each forward."""
        dev = torch.device(device)
        comp = torch.cuda.current_stream(dev)
        keys = ("x3", "x2", "x1", "hist_data", "mask")
        # streams, device staging buffers and pinned result buffers persist across calls (pinned
        # allocation costs tens of ms and synchronises the device; it must not sit in a hot loop)
        cache = self.__dict__.setdefault("_stream_cache", {})
        if (str(dev), depth) not in cache:
            cache[(str(dev), depth)] = dict(
                h2d=torch.cuda.Stream(dev), d2h=torch.cuda.Stream(dev),
                slots=[dict(inp=None, out=None, comp_done=torch.cuda.Event(),
                            out_ready=torch.cuda.Event(), busy=False, graph=None,
                            # per-input / per-level events (external: they survive CUDA-graph capture as event nodes)
                            ready={k: torch.cuda.Event(external=True) for k in ("hist", "x3", "x2", "x1")},
                            done=[torch.cuda.Event(external=True) for _ in range(3)]) for _ in range(depth)])
        st = cache[(str(dev), depth)]
        h2d, d2h, slots = st["h2d"], st["d2h"], st["slots"]
        for sl in slots:
            sl["busy"] = False
        pending: List[Tuple[int, int]] = []            # (batch index, slot)
        seed_it = iter(seeds) if seeds is not None else None

        def drain(idx_slot):
            idx, si = idx_slot
            slots[si]["out_ready"].synchronize()
            return idx, slots[si]["out"]

        for i, hb in enumerate(batches):
            si = i % depth
            sl = slots[si]
            if sl["busy"]:                               # slot still owned by batch i-depth: hand it out first
                yield drain(pending.pop(0))
                sl["busy"] = False
            if sl["inp"] is None or any(sl["inp"][k].shape != hb[k].shape or sl["inp"][k].dtype != hb[k].dtype for k in keys):
                sl["inp"] = {k: torch.empty(hb[k].shape, dtype=hb[k].dtype, device=dev) for k in keys}
                sl["graph"] = None
            with torch.cuda.stream(h2d):
                h2d.wait_event(sl["comp_done"])          # previous compute on these input buffers finished
                # smallest first: histograms + mask, then the 1/16, 1/8, 1/4 maps - each followed by its own event, so that a
                # level starts when ITS map has landed (the first batch of a run no longer waits for all 100 MB)
                for k in ("hist_data", "mask"):
                    sl["inp"][k].copy_(hb[k], non_blocking=True)
                sl["ready"]["hist"].record(h2d)
                for k in ("x3", "x2", "x1"):
                    sl["inp"][k].copy_(hb[k], non_blocking=True)
                    sl["ready"][k].record(h2d)
            # per-input / per-level events rather than one of each per batch: measured K = 10 16.50 -> 16.92 k frames/s
            ev = dict(ready=sl["ready"], done=sl["done"])
            if seed_it is not None:
                torch.manual_seed(next(seed_it))
            d = sl["inp"]
            if graph:                                    # one captured forward per slot (its device buffers are the static inputs)
                if sl.get("graph") is None:
                    comp.synchronize()                   # capture replays the forward: the slot's first inputs must have landed
                    h2d.synchronize()                    # ... all of them (with per-level events `comp` does not wait for h2d)
                    sl["graph"] = self.make_graphed(d["x3"], d["x2"], d["x1"], d["hist_data"], d["mask"], patch_info, copy_inputs=False, **ev)
                outs = sl["graph"]()
            else:
                outs = self.forward(d["x3"], d["x2"], d["x1"], d["hist_data"], d["mask"], patch_info, **ev)
            sl["comp_done"].record(comp)
            if sl["out"] is None or any(p.shape != o.shape or p.dtype != o.dtype for p, o in zip(sl["out"], outs)):
                sl["out"] = [torch.empty(o.shape, dtype=o.dtype, pin_memory=True) for o in outs]
            with torch.cuda.stream(d2h):
                for j, (p, o) in enumerate(zip(sl["out"], outs)):
                    d2h.wait_event(sl["done"][j])         # this level's map is complete (the others may still be running)
                    p.copy_(o, non_blocking=True)
                sl["out_ready"].record(d2h)
            # keep the device results referenced until this slot is drained (host-synchronised on out_ready):
            # record_stream() would instead park the blocks in the allocator until an event query succeeds,
            # and the resulting occasional cudaMalloc stalls the device for ~100 ms
            sl["dev_out"] = outs
            sl["busy"] = True
            pending.append((i, si))
        while pending:
            yield drain(pending.pop(0))
