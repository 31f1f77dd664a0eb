"""Thin object layer over the C ABI: one ``Device`` (nxfx_ctx) per GPU per process, device
buffers and pinned host arrays.  PETSc ``Vec``/``Mat`` stand-ins in ``la.py`` are built on these."""

from __future__ import annotations

import ctypes as C
import weakref

import numpy as np

from . import _lib


class Device:
    """Owner of an ``nxfx_ctx``.  ``call(name, *args)`` raises RuntimeError with the library's
    message on any non-zero status (never a silent fallback)."""

    def __init__(self, index: int = 0, stream: int | None = None):
        self.lib = _lib.load()
        handle = C.c_void_p()
        rc = self.lib.nxfx_create(C.byref(handle), int(index))
        if rc != 0 or not handle:
            raise RuntimeError(
                f"nxfx_create(device={index}) failed with status {rc}: no usable CUDA device. "
                "networks_fenicsx_b200 has no CPU fallback."
            )
        self.handle = handle
        self.index = int(index)
        self._finalizer = weakref.finalize(self, self.lib.nxfx_destroy, handle)
        self.stream = None  # cudaStream_t of the ctx as an int; None: the legacy default stream
        self._torch_stream = None
        if stream is not None:
            self.set_stream(stream)

    def set_stream(self, stream: int | None) -> None:
        """Run the ctx on ``stream`` (a ``cudaStream_t`` as an int; None or 0: the legacy default stream)."""
        self.call("nxfx_set_stream", C.c_void_p(stream or None))
        self.stream = int(stream) if stream else None
        self._torch_stream = None

    def call(self, name: str, *args) -> None:
        rc = getattr(self.lib, name)(self.handle, *args)
        if rc != 0:
            msg = self.lib.nxfx_last_error(self.handle)
            raise RuntimeError(f"{name} failed ({rc}): {msg.decode() if msg else ''}")

    def sync(self) -> None:
        self.call("nxfx_sync")

    @property
    def launch_count(self) -> int:
        return int(self.lib.nxfx_launch_count(self.handle))

    def timer_start(self) -> None:
        self.call("nxfx_timer_start")

    def timer_stop(self) -> float:
        ms = C.c_double()
        self.call("nxfx_timer_stop", C.byref(ms))
        return ms.value

    # ---- ordering against torch (CUDA tensors handed in or out) ----------------------------------
    def torch_stream(self):
        """The ctx's stream as a ``torch.cuda.Stream``."""
        import torch  # noqa: PLC0415

        if self._torch_stream is None:
            cuda = torch.device("cuda", self.index)
            self._torch_stream = (torch.cuda.ExternalStream(self.stream, device=cuda) if self.stream
                                  else torch.cuda.default_stream(cuda))
        return self._torch_stream

    def wait_for_torch(self, *tensors) -> None:
        """Order the work this ctx enqueues next after what the current torch stream has enqueued so far (an
        event, no host wait), and keep torch's caching allocator from handing ``tensors`` to a new tensor before
        the ctx's stream has passed that work (``record_stream``)."""
        import torch  # noqa: PLC0415

        lib = self.torch_stream()
        cur = torch.cuda.current_stream(lib.device)
        if cur.cuda_stream != lib.cuda_stream:
            lib.wait_stream(cur)
        for t in tensors:
            t.record_stream(lib)

    def torch_wait(self) -> None:
        """Order the work the current torch stream enqueues next after what this ctx has enqueued so far."""
        import torch  # noqa: PLC0415

        lib = self.torch_stream()
        cur = torch.cuda.current_stream(lib.device)
        if cur.cuda_stream != lib.cuda_stream:
            cur.wait_stream(lib)

    def empty(self, n: int, dtype=np.float64) -> "DeviceArray":
        return DeviceArray(self, int(n), np.dtype(dtype))

    def from_host(self, a: np.ndarray) -> "DeviceArray":
        a = np.ascontiguousarray(a)
        d = DeviceArray(self, a.size, a.dtype)
        d.upload(a)
        return d

    def pinned(self, n: int, dtype=np.float64) -> np.ndarray:
        """Pinned host ndarray (freed when garbage collected)."""
        dtype = np.dtype(dtype)
        ptr = C.c_void_p()
        nbytes = max(int(n) * dtype.itemsize, 8)
        self.call("nxfx_host_alloc", C.c_size_t(nbytes), C.byref(ptr))
        buf = (C.c_char * nbytes).from_address(ptr.value)
        arr = np.frombuffer(buf, dtype=dtype, count=int(n))
        weakref.finalize(buf, self.lib.nxfx_host_free, self.handle, ptr)
        return arr


_default_devices: dict[int, Device] = {}


def default_device(index: int = 0) -> Device:
    if index not in _default_devices:
        _default_devices[index] = Device(index)
    return _default_devices[index]


class DeviceArray:
    """Flat device buffer of ``n`` elements.  ``on_write`` (optional) is called after every write this
    object or a view of it makes (``upload``, ``zero``): the owner of a borrowed buffer learns that its
    contents changed (``Mat.values``: ``Mat.touch``).

    ``__cuda_array_interface__`` (version 3) exposes the buffer without a copy, e.g. ``torch.as_tensor(a,
    device="cuda")``; the tensor keeps this object, and so the memory, alive.  ``shape`` / ``strides`` (bytes)
    describe a strided view of the buffer (default: the ``n`` elements, contiguous).  The interface names the
    ctx's stream; the Python layer itself orders the ctx's stream against torch's current stream with events
    (:meth:`Device.wait_for_torch`, :meth:`Device.torch_wait`), since torch does not read that field."""

    def __init__(self, dev: Device, n: int, dtype=np.float64, ptr: int | None = None, on_write=None,
                 shape: tuple | None = None, strides: tuple | None = None):
        self.dev = dev
        self.n = int(n)
        self.dtype = np.dtype(dtype)
        self.owned = ptr is None
        self.on_write = on_write
        self.shape = (self.n,) if shape is None else tuple(int(s) for s in shape)
        self.strides = None if strides is None else tuple(int(s) for s in strides)
        if ptr is None:
            p = C.c_void_p()
            dev.call("nxfx_malloc", C.c_size_t(self.nbytes), C.byref(p))
            self.ptr = p.value
            self._finalizer = weakref.finalize(self, dev.lib.nxfx_free, dev.handle, C.c_void_p(self.ptr))
        else:
            self.ptr = int(ptr)

    @property
    def nbytes(self) -> int:
        return self.n * self.dtype.itemsize

    @property
    def c_ptr(self) -> C.c_void_p:
        return C.c_void_p(self.ptr)

    @property
    def __cuda_array_interface__(self) -> dict:
        # stream: 1 = the legacy default stream (0 is not allowed by the protocol)
        return {"shape": self.shape, "typestr": self.dtype.str, "data": (self.ptr, False), "version": 3,
                "strides": self.strides, "stream": self.dev.stream or 1}

    def as_tensor(self):
        """Zero-copy ``torch.Tensor`` on the ctx's device over this buffer (through ``__cuda_array_interface__``)."""
        import torch  # noqa: PLC0415

        return torch.as_tensor(self, device=torch.device("cuda", self.dev.index))

    def upload(self, host: np.ndarray, sync: bool = True) -> None:
        host = np.ascontiguousarray(host, dtype=self.dtype)
        assert host.size == self.n, (host.size, self.n)
        if self.n:
            self.dev.call("nxfx_memcpy_h2d", self.c_ptr, C.c_void_p(host.ctypes.data), C.c_size_t(self.nbytes))
        if sync:
            self.dev.sync()
        if self.on_write is not None:
            self.on_write()

    def download(self, out: np.ndarray | None = None, sync: bool = True) -> np.ndarray:
        if out is None:
            out = np.empty(self.n, dtype=self.dtype)
        assert out.size == self.n and out.dtype == self.dtype and out.flags.c_contiguous
        if self.n:
            self.dev.call("nxfx_memcpy_d2h", C.c_void_p(out.ctypes.data), self.c_ptr, C.c_size_t(self.nbytes))
        if sync:
            self.dev.sync()
        return out

    def zero(self) -> None:
        if self.n:
            self.dev.call("nxfx_memset", self.c_ptr, 0, C.c_size_t(self.nbytes))
        if self.on_write is not None:
            self.on_write()

    def view(self, offset: int, n: int) -> "DeviceArray":
        assert 0 <= offset and offset + n <= self.n
        v = DeviceArray(self.dev, n, self.dtype, ptr=self.ptr + offset * self.dtype.itemsize, on_write=self.on_write)
        v._keepalive = self
        return v
