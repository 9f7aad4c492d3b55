"""Torch plumbing shared by the ctypes faces of the library's MLP handles: ``ppo.FusedUpdate`` (include/dnppo.h) and
``sac.FusedSACActor`` (include/dnsac.h).  Kept apart from ``_lib`` so that the ctypes binding does not import torch."""
from __future__ import annotations

import ctypes as C
import types

import torch
import torch.distributed as dist

from . import _lib as L


def world() -> int:
    return dist.get_world_size() if dist.is_available() and dist.is_initialized() else 1


def flat_views(flat: torch.Tensor, like) -> list:
    """Consecutive views of `flat`, one per tensor of `like` and shaped like it, from element 0 on."""
    views, off = [], 0
    for t in like:
        views.append(flat[off:off + t.numel()].view_as(t))
        off += t.numel()
    return views


def offsets(named_parameters) -> dict:
    """name -> element offset of that parameter in a flat vector that holds the parameters one after another."""
    offs, off = {}, 0
    for name, p in named_parameters:
        offs[name], off = off, off + p.numel()
    return offs


def sm100(device) -> bool:
    """A compute-capability-10 CUDA device: the only kind the library's MLP kernels are built for."""
    dev = torch.device(device)
    return dev.type == "cuda" and torch.cuda.get_device_capability(dev)[0] == 10


def widths_ok(arch, obs_dim: int) -> bool:
    """The hidden layers and observation width every MLP handle accepts: 1..4 hidden layers, each a multiple of 128 between 128
    and 512, and 1 <= obs_dim <= 64 (one padded 64-column k-block)."""
    arch = tuple(arch)
    return 1 <= len(arch) <= 4 and all(w % 128 == 0 and 128 <= w <= 512 for w in arch) and 1 <= obs_dim <= 64


class Handle:
    """One library handle on ``self.device``, created and called with that device current and on its current stream.
    ``ABI`` is the entry-point prefix: ``<ABI>_create``, ``_destroy``, ``_sync_weights`` and ``_buffer``."""

    ABI = ""

    def __init__(self, device):
        self.L, self.lib = L, L.lib()
        self.device = device
        self.handle = C.c_void_p()

    def _create(self, cfg, *ptrs):
        """``<ABI>_create(&cfg, device index, *ptrs, &handle)`` after the device's pending work (which may still write the
        parameters) has finished."""
        self.cfg_c = cfg
        name = self.ABI + "_create"
        with torch.cuda.device(self.device):
            torch.cuda.synchronize(self.device)
            L.check(getattr(self.lib, name)(C.byref(cfg), self.device.index or 0, *ptrs, C.byref(self.handle)), name)

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def call(self, name: str, *args):
        """``name(handle, *args, stream)``; raises ``_lib.DroneNavError`` when it fails."""
        with torch.cuda.device(self.device):
            self.L.check(getattr(self.lib, name)(self.handle, *args, self._stream()), name)

    def sync_weights(self):
        """FP32 parameters -> the BF16 weight planes the kernels read."""
        self.call(self.ABI + "_sync_weights")

    def close(self):
        if getattr(self, "handle", None):
            getattr(self.lib, self.ABI + "_destroy")(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:  # noqa: BLE001
            pass

    def _raw_buffer(self, name: str, typestr: str) -> torch.Tensor:
        """An internal allocation of the handle (``<ABI>_buffer``), as a flat tensor viewing the library's memory."""
        ptr, elems = C.c_void_p(), C.c_int64()
        fn = self.ABI + "_buffer"
        self.L.check(getattr(self.lib, fn)(self.handle, name.encode(), C.byref(ptr), C.byref(elems)), fn)
        view = types.SimpleNamespace(__cuda_array_interface__={"shape": (elems.value,), "typestr": typestr,
                                                               "data": (ptr.value, False), "version": 2})
        return torch.as_tensor(view, device=self.device)
