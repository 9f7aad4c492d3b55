"""Torch plumbing shared by the PPO and SAC learners: the ctypes faces of the library's MLP handles (``ppo.FusedUpdate``,
include/dnppo.h, and ``sac.FusedSACActor``, include/dnsac.h) and the CUDA-graph capture of the update steps and of the trainers'
collection phases.  Kept apart from ``_lib`` so that the ctypes binding does not import torch."""
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


def capture_graphs(stages, warmup, tensors, optimizers, device) -> list:
    """One CUDA graph per callable of `stages`, all from one shared memory pool (a stage may consume tensors an earlier stage
    produced), captured after ``warmup()`` has run on a side stream (lazy kernel loading, allocator, library workspaces,
    optimiser state).  The warm-up takes real steps, so afterwards every tensor of `tensors` and the state of every optimiser
    of `optimizers` is put back bit for bit, in place (the graphs bake those pointers in); optimiser state the warm-up
    created ends zeroed, which is a fresh Adam state.  Every rank of a data-parallel job must run the same warm-up."""
    opt_state = lambda: [v for o in optimizers for st in o.state.values() for v in st.values() if torch.is_tensor(v)]
    saved = [(t, t.detach().clone()) for t in list(tensors) + opt_state()]
    side = torch.cuda.Stream(device=device)
    side.wait_stream(torch.cuda.current_stream(device))
    quiet = getattr(torch.autograd.graph, "set_warn_on_accumulate_grad_stream_mismatch", None)
    if quiet is not None:        # the gradient buckets were created on the current stream, the warm-up runs on a side stream: intended
        quiet(False)
    with torch.cuda.stream(side):
        warmup()
    torch.cuda.current_stream(device).wait_stream(side)
    with torch.no_grad():
        for v in opt_state():
            v.zero_()
        for t, s in saved:
            t.copy_(s)
    pool = torch.cuda.graph_pool_handle()
    graphs = []
    for stage in stages:
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, pool=pool):
            stage()
        graphs.append(g)
    return graphs


class PhaseGraph:
    """A phase of a trainer (a callable that issues the same launches every time) run from a CUDA graph: the first call launches
    it (loading every kernel), the next call captures and replays it, later calls with the same key replay.  A new key captures
    again, without another launched call.  A call with ``enabled`` false launches."""

    def __init__(self):
        self.key, self.graph, self.warm = None, None, False

    def run(self, enabled: bool, key, phase) -> None:
        if not (enabled and self.warm):
            phase()
            self.warm = True
            return
        if self.graph is None or self.key != key:
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                phase()
            self.key, self.graph = key, g
        self.graph.replay()


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
