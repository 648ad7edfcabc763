"""Host-side weight packing for libcfp.

The kernels want nn.Linear / conv weights transposed to [in][out] fp32 with
eval-mode BatchNorm folded in, and bf16 UMMA blocks for the tensor-core engine.
Packing is a one-off per parameter version (cached) and it is plumbing, not part
of the timed hot path.  It runs on the HOST: every parameter is read back once
(plain device->host copies), the packed tensors are laid out in one flat byte
buffer and reach the device with ONE host->device copy per module - no ATen
kernel is launched for it (round 1 packed with torch ops on the device: ~970
copy / cast launches before the first libcfp kernel, which is all a profiler's
launch window then showed).
"""
from __future__ import annotations

import torch
import torch.nn as nn


import ctypes as C
import threading


def host(t: torch.Tensor) -> torch.Tensor:
    """Parameter / buffer -> detached fp32 CPU tensor (device->host copy in the storage dtype, cast on the host)."""
    return t.detach().cpu().float()


def fold_bn(bn: nn.modules.batchnorm._BatchNorm):
    """Eval-mode BN as y = x*scale + shift (fp32, host)."""
    scale = host(bn.weight) * torch.rsqrt(host(bn.running_var) + bn.eps)
    shift = host(bn.bias) - host(bn.running_mean) * scale
    return scale, shift


def linear_t(lin_weight: torch.Tensor) -> torch.Tensor:
    """nn.Linear weight [out,in] -> [in,out] fp32 contiguous (host)."""
    return host(lin_weight).t().contiguous()


def umma_block(w: torch.Tensor, dtype: torch.dtype = torch.bfloat16) -> torch.Tensor:
    """[N,K] weight -> 16-bit block in the canonical K-major no-swizzle UMMA layout
    [K/8][N][8] (csrc/umma.cuh): element (n,k) at ((k//8)*N + n)*8 + k%8."""
    n, k = w.shape
    assert k % 8 == 0
    return w.detach().cpu().to(dtype).contiguous().view(n, k // 8, 8).permute(1, 0, 2).contiguous()


class Packer(list):
    """The packed tensors of one module, in packing order (a list of host tensors), and their places in one flat
    byte buffer.  ``ref(t)`` hands out t's byte offset - what the weight structs of include/cfp.h hold until
    ``upload()`` has copied the buffer to the device and ``relocate()`` has turned the offsets into device pointers.
    Offsets start at ALIGN, so that 0 stays the null pointer."""
    ALIGN = 256

    def __init__(self):
        super().__init__()
        self._offsets = {}
        self._size = self.ALIGN

    def ref(self, t: torch.Tensor) -> int:
        key = id(t)
        if key not in self._offsets:
            if not any(t is x for x in self):
                self.append(t)
            if t.device.type != "cpu" or not t.is_contiguous():
                raise ValueError("packed tensors are contiguous host tensors")
            self._offsets[key] = self._size
            nbytes = t.numel() * t.element_size()
            self._size += (nbytes + self.ALIGN - 1) // self.ALIGN * self.ALIGN
        return self._offsets[key]

    def upload(self, device) -> torch.Tensor:
        """One flat uint8 buffer on ``device`` holding every referenced tensor (one host->device copy)."""
        flat = torch.zeros(self._size, dtype=torch.uint8)
        for t in self:
            off = self._offsets.get(id(t))
            if off is not None and t.numel():
                flat[off:off + t.numel() * t.element_size()] = t.reshape(-1).view(torch.uint8)
        return flat.to(device)


def relocate(struct, base: int):
    """Add ``base`` to every non-null pointer field of a (nested) ctypes weight struct, in place."""
    for name, typ in struct._fields_:
        val = getattr(struct, name)
        if typ is C.c_void_p:
            if val:
                setattr(struct, name, val + base)
        elif isinstance(val, C.Structure):
            relocate(val, base)
        elif isinstance(val, C.Array) and val._type_ is C.c_void_p:
            for i in range(len(val)):
                if val[i]:
                    val[i] = val[i] + base
    return struct


class PackCache:
    """Re-pack only when a parameter / buffer of the CALLING module changed (in-place update, load_state_dict,
    .to(device)).  The cache is keyed by the calling module's own tensors: ``nn.DataParallel`` replicas share their
    original's ``__dict__`` entries, so a cache that looked at the module it was created for would hand device-0
    weight pointers to every replica.  Replicas (re-created by DataParallel on every forward, parameters re-broadcast)
    are never cached: they pack on each call and the packed buffer lives as long as the call's kernels need it
    (stream-ordered reuse by torch's allocator)."""

    def __init__(self, module: nn.Module = None):
        self._lock = threading.Lock()
        self._entries = {}                       # device -> (key, value)
        self.generation = 0                      # bumped whenever a packed copy is dropped or replaced

    def __deepcopy__(self, memo):                # a copied / unpickled module starts with an empty cache
        return PackCache()

    def __reduce__(self):
        return (PackCache, ())

    def invalidate(self):
        """Drop every packed copy: for writers that update parameters through raw pointers (the libcfp optimizer step,
        cfpnet_b200/train.py), which torch's version counters do not see."""
        with self._lock:
            self._entries.clear()
            self.generation += 1

    def held(self) -> list:
        """The packed copies this cache holds now (a CUDA graph that reads them keeps them alive with this list)."""
        with self._lock:
            return list(self._entries.values())

    @staticmethod
    def _key(module: nn.Module):
        return tuple((t.data_ptr(), t._version, str(t.device)) for t in
                     list(module.parameters()) + list(module.buffers()))

    def get(self, module: nn.Module, build):
        if getattr(module, "_is_replica", False):
            with torch.no_grad():
                return build()
        key = self._key(module)
        dev = key[0][2] if key else "cpu"
        with self._lock:
            hit = self._entries.get(dev)
            if hit is None or hit[0] != key:
                with torch.no_grad():
                    hit = (key, build())
                self._entries[dev] = hit
                self.generation += 1
            return hit[1]


class Scratch:
    """Per-device scratch tensors owned by a module (workspace + token map), reused across calls on one stream.
    One entry per device; a module shared by several threads (``nn.DataParallel``'s original module is only ever run
    on device 0, replicas get their own Scratch) never sees another device's entry dropped under it."""

    def __init__(self):
        self._lock = threading.Lock()
        self._entries = {}                       # device index -> (key, tensors)

    def __deepcopy__(self, memo):
        return Scratch()

    def __reduce__(self):
        return (Scratch, ())

    def held(self) -> list:
        """The scratch tensors this module holds now (see PackCache.held)."""
        with self._lock:
            return list(self._entries.values())

    def get(self, device_index, key, fits, make):
        with self._lock:
            hit = self._entries.get(device_index)
            if hit is None or hit[0] != key or not fits(hit[1]):
                self._entries.pop(device_index, None)      # free the old entry before allocating its replacement
                hit = (key, make())
                self._entries[device_index] = hit
            return hit[1]
