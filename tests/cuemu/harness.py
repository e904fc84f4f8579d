"""Run the product's Python binding (mmssl_b200/_lib.py and the modules above it) against the host-emulated library
(tests/cuemu/_build/libmmssl_emu.so) -- TEST INFRASTRUCTURE ONLY.

``emulated_device(monkeypatch)`` makes, for the duration of one test:
  * ``_lib.load()`` return the emulated library (same C ABI, same ctypes signatures, host pointers as "device" pointers);
  * ``tensor.cuda()`` a plain copy, ``tensor.is_cuda`` true, ``torch.cuda.synchronize`` a no-op,
    the stream argument NULL.
The bodies of the ``-m gpu`` tests can then be executed unchanged on the CPU: same wrappers, same argument marshalling,
same kernels (compiled from the same .cu sources), CUDA's block / warp semantics provided by the fiber emulator.
The patches are undone by ``monkeypatch``; nothing under mmssl_b200/ knows about this."""
import contextlib
import ctypes as C
import os
import weakref

import torch

from . import build as _build

_EMU = None


def emu_lib():
    global _EMU
    if _EMU is None:
        from mmssl_b200 import _lib
        lib = C.CDLL(_build.build())
        have = []
        for name, (res, args) in _lib._SIGS.items():
            try:
                fn = getattr(lib, name)
            except AttributeError:
                continue                      # entry points of files the emulator cannot compile (CUB, TMA, tcgen05)
            fn.restype, fn.argtypes = res, args
            have.append(name)
        lib._emulated = tuple(have)
        _EMU = lib
    return _EMU


def set_order(order: str) -> None:
    """fwd | rev | shuffle:<seed> -- the order in which the fibers of a block get the CPU.  CUEMU_ORDER_FORCE overrides the
    tests' own choice (to sweep the whole emulated suite under another thread order)."""
    os.environ["CUEMU_ORDER"] = os.environ.get("CUEMU_ORDER_FORCE", order)


class _NullStream:
    """torch.cuda.Stream stand-in: the emulator executes every launch synchronously, in program order."""
    cuda_stream = 0

    def __init__(self, *a, **k):
        pass

    def wait_stream(self, other):
        pass

    def synchronize(self):
        pass


def _on_cpu(fn):
    """torch factory with ``device="cuda"`` rewritten to the CPU (the tests' inputs are created on the 'device')."""
    def wrapped(*a, **k):
        if "device" in k and k["device"] is not None and str(k["device"]).startswith("cuda"):
            k["device"] = "cpu"
        return fn(*a, **k)
    wrapped.__name__ = getattr(fn, "__name__", "factory")
    return wrapped


class _Guard:
    """Red zones around every tensor the patched factories hand out; ``check`` runs after every library call.
    The "device" is the host heap here, so an out-of-bounds kernel write would otherwise corrupt it silently."""
    PAD = 512

    def __init__(self, real_empty):
        self.real_empty, self.live = real_empty, []

    def alloc(self, shape, dtype, fill):
        n = 1
        for v in shape:
            n *= int(v)
        es = self.real_empty(0, dtype=dtype).element_size()
        buf = self.real_empty(n * es + 2 * self.PAD, dtype=torch.uint8)
        buf[:self.PAD] = 0xA5
        buf[self.PAD + n * es:] = 0xA5
        view = buf[self.PAD:self.PAD + n * es].view(dtype).reshape(tuple(shape)) if n else self.real_empty(tuple(shape), dtype=dtype)
        if fill is not None and n:
            view.fill_(fill)
        if n:
            self.live.append((weakref.ref(view), buf, tuple(shape), dtype))
        return view

    def check(self, where):
        keep = []
        for ref, buf, shape, dtype in self.live:
            if ref() is None:
                continue
            keep.append((ref, buf, shape, dtype))
            lo, hi = buf[:self.PAD], buf[buf.numel() - self.PAD:]
            if bool((lo != 0xA5).any()) or bool((hi != 0xA5).any()):
                side = "before" if bool((lo != 0xA5).any()) else "after"
                raise AssertionError(f"cuemu guard: {where} wrote {side} a {dtype} tensor of shape {shape}")
        self.live = keep


class _Checked:
    """Library proxy: every call is followed by a red-zone check."""

    def __init__(self, lib, guard):
        object.__setattr__(self, "_lib", lib)
        object.__setattr__(self, "_guard", guard)

    def __getattr__(self, name):
        fn = getattr(self._lib, name)
        if not callable(fn):
            return fn
        guard = self._guard

        def call(*a):
            r = fn(*a)
            guard.check(name)
            return r
        return call


def emulated_device(monkeypatch, guard: bool = False):
    from mmssl_b200 import _lib
    guard = guard or os.environ.get("CUEMU_GUARD") == "1"       # CUEMU_GUARD=1 pytest ... : the whole emulated suite with red zones
    lib = emu_lib()
    # a failed launch leaves a sticky error in the emulator, like CUDA: clear it between tests
    clear = getattr(lib, "cuemu_clear_error", None)
    if clear is not None:
        clear()
    monkeypatch.setattr(_lib, "load", lambda require_device=False: lib)
    monkeypatch.setattr(_lib, "_lib", lib)
    # the NULL stream comes from the patched torch.cuda.current_stream, which _lib.stream() reads at every call.  Patching
    # `stream` in the modules instead would leak: a module first imported during the test keeps the patched function it
    # imported, and on a machine with a GPU its later launches would bypass the current stream (and any graph capture on it).
    monkeypatch.setattr(torch.Tensor, "cuda", lambda self, *a, **k: self.clone())   # a copy, like a real host->device transfer
    real_to = torch.Tensor.to

    def to(self, *a, **k):
        is_cuda = lambda d: isinstance(d, (str, torch.device)) and str(d).startswith("cuda")
        a = tuple("cpu" if is_cuda(x) else x for x in a)
        if is_cuda(k.get("device")):
            k["device"] = "cpu"
        return real_to(self, *a, **k)
    monkeypatch.setattr(torch.Tensor, "to", to)
    monkeypatch.setattr(torch.Tensor, "is_cuda", property(lambda self: True))
    monkeypatch.setattr(torch.cuda, "synchronize", lambda *a, **k: None)
    monkeypatch.setattr(torch.cuda, "Stream", _NullStream)
    monkeypatch.setattr(torch.cuda, "current_stream", lambda *a, **k: _NullStream())
    monkeypatch.setattr(torch.cuda, "stream", lambda s: contextlib.nullcontext())
    if guard:
        g = _Guard(torch.empty)
        lib = _Checked(lib, g)
        monkeypatch.setattr(_lib, "load", lambda require_device=False: lib)
        monkeypatch.setattr(_lib, "_lib", lib)

        def factory(fill):
            def make(*shape, dtype=torch.float32, device=None, **kw):
                if len(shape) == 1 and isinstance(shape[0], (tuple, list, torch.Size)):
                    shape = tuple(shape[0])
                return g.alloc(shape, dtype or torch.float32, fill)
            return make
        monkeypatch.setattr(torch, "empty", factory(None))
        monkeypatch.setattr(torch, "zeros", factory(0))
        monkeypatch.setattr(torch, "ones", factory(1))
        monkeypatch.setattr(torch, "empty_like", lambda t, **kw: g.alloc(tuple(t.shape), kw.get("dtype") or t.dtype, None))
        monkeypatch.setattr(torch, "zeros_like", lambda t, **kw: g.alloc(tuple(t.shape), kw.get("dtype") or t.dtype, 0))
    for fname in ("randn", "rand", "randint", "zeros", "ones", "empty", "full", "tensor", "arange", "as_tensor", "randperm"):
        monkeypatch.setattr(torch, fname, _on_cpu(getattr(torch, fname)))
    return lib
