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
        if stream is not None:
            self.call("nxfx_set_stream", C.c_void_p(stream))

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
    contents changed (``Mat.values``: ``Mat.touch``)."""

    def __init__(self, dev: Device, n: int, dtype=np.float64, ptr: int | None = None, on_write=None):
        self.dev = dev
        self.n = int(n)
        self.dtype = np.dtype(dtype)
        self.owned = ptr is None
        self.on_write = on_write
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
