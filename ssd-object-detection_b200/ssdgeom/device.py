"""Device memory for the host layer: a small owning array type over ssdg_device_alloc plus
zero-copy views of anything that exposes ``__cuda_array_interface__`` (torch CUDA tensors do).
No torch import here -- PyTorch is optional plumbing for callers, not a dependency."""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _native as N


class Stream:
    """Owning CUDA stream (non-blocking)."""

    def __init__(self, priority=None):
        """priority: None (default), or "high" / "low" (the device's extreme stream priorities)."""
        if priority not in (None, "high", "low"):
            raise ValueError("stream priority must be None, 'high' or 'low', not %r" % (priority,))
        h = C.c_void_p()
        if priority is None:
            N.check(N.lib().ssdg_stream_create(C.byref(h)), "stream_create")
        else:
            N.check(N.lib().ssdg_stream_create_priority(C.byref(h), 1 if priority == "high" else 0), "stream_create")
        self.handle = h.value

    def sync(self):
        N.check(N.lib().ssdg_stream_sync(self.handle), "stream_sync")

    def __del__(self):
        try:
            if self.handle:
                N.lib().ssdg_stream_destroy(self.handle)
        except Exception:
            pass


def stream_handle(stream) -> int | None:
    """None -> legacy default stream; Stream; int; or a torch.cuda.Stream (has .cuda_stream)."""
    if stream is None:
        return None
    if isinstance(stream, Stream):
        return stream.handle
    if hasattr(stream, "cuda_stream"):
        return int(stream.cuda_stream) or None
    return int(stream) or None


def current_device() -> int:
    d = C.c_int(0)
    N.check(N.lib().ssdg_get_device(C.byref(d)), "get_device")
    return d.value


def sync(stream=None):
    N.check(N.lib().ssdg_stream_sync(stream_handle(stream)), "stream_sync")


class Event:
    def __init__(self):
        h = C.c_void_p()
        N.check(N.lib().ssdg_event_create(C.byref(h)), "event_create")
        self.handle = h.value

    def record(self, stream=None):
        N.check(N.lib().ssdg_event_record(self.handle, stream_handle(stream)), "event_record")

    def elapsed_ms(self, later: "Event") -> float:
        ms = C.c_float(0)
        N.check(N.lib().ssdg_event_elapsed_ms(self.handle, later.handle, C.byref(ms)), "event_elapsed")
        return ms.value

    def __del__(self):
        try:
            if self.handle:
                N.lib().ssdg_event_destroy(self.handle)
        except Exception:
            pass


def stream_wait_event(stream, event: Event):
    N.check(N.lib().ssdg_stream_wait_event(stream_handle(stream), event.handle), "stream_wait_event")


class DeviceArray:
    """Contiguous device buffer with a shape and dtype.  Owns its memory unless ``owner`` is
    given (then it is a view that keeps ``owner`` alive)."""

    def __init__(self, shape, dtype, ptr=None, owner=None):
        self.shape = tuple(int(s) for s in (shape if isinstance(shape, (tuple, list)) else (shape,)))
        self.dtype = np.dtype(dtype)
        self.nbytes = int(np.prod(self.shape, dtype=np.int64)) * self.dtype.itemsize
        self._owner = owner
        self._owned = ptr is None
        if ptr is None:
            h = C.c_void_p()
            N.check(N.lib().ssdg_device_alloc(C.byref(h), max(self.nbytes, 1)), "device_alloc")
            ptr = h.value
        self.ptr = int(ptr)

    @property
    def size(self):
        return int(np.prod(self.shape, dtype=np.int64))

    @property
    def __cuda_array_interface__(self):
        return {"shape": self.shape, "typestr": self.dtype.str, "data": (self.ptr, False), "version": 3,
                "strides": None}

    def __del__(self):
        try:
            if self._owned and self.ptr:
                N.lib().ssdg_device_free(self.ptr)
                self.ptr = 0
        except Exception:
            pass

    def copy_from_host(self, arr: np.ndarray, stream=None):
        arr = np.ascontiguousarray(arr, dtype=self.dtype)
        assert arr.nbytes == self.nbytes, "size mismatch"
        N.check(N.lib().ssdg_memcpy_h2d(self.ptr, arr.ctypes.data, self.nbytes, stream_handle(stream)), "h2d")
        self._keep = arr  # keep the source alive until the (possibly async) copy has run
        return self

    def to_host(self, stream=None, out: np.ndarray | None = None) -> np.ndarray:
        if out is None:
            out = np.empty(self.shape, dtype=self.dtype)
        N.check(N.lib().ssdg_memcpy_d2h(out.ctypes.data, self.ptr, self.nbytes, stream_handle(stream)), "d2h")
        sync(stream)
        return out

    def zero_(self, stream=None):
        N.check(N.lib().ssdg_memset(self.ptr, 0, self.nbytes, stream_handle(stream)), "memset")
        return self

    def view(self, shape, dtype=None):
        v = DeviceArray(shape, dtype or self.dtype, ptr=self.ptr, owner=self)
        assert v.nbytes <= self.nbytes
        return v


def empty(shape, dtype) -> DeviceArray:
    return DeviceArray(shape, dtype)


def to_device(arr, dtype=None, stream=None) -> DeviceArray:
    arr = np.ascontiguousarray(arr, dtype=dtype)
    return DeviceArray(arr.shape, arr.dtype).copy_from_host(arr, stream)


def is_device(x) -> bool:
    return hasattr(x, "__cuda_array_interface__")


def as_device(x, dtype=None, stream=None) -> DeviceArray:
    """Device view of ``x``: zero-copy for CUDA arrays (dtype must already match and the array
    must be contiguous), upload for host arrays."""
    if isinstance(x, DeviceArray):
        if dtype is not None and np.dtype(dtype) != x.dtype:
            raise TypeError("device array has dtype %s, expected %s" % (x.dtype, np.dtype(dtype)))
        return x
    if is_device(x):
        cai = x.__cuda_array_interface__
        dt = np.dtype(cai["typestr"])
        if dtype is not None and np.dtype(dtype) != dt:
            raise TypeError("device array has dtype %s, expected %s" % (dt, np.dtype(dtype)))
        if cai.get("strides") is not None:
            expect = np.empty(cai["shape"], dtype=dt).strides
            if tuple(cai["strides"]) != tuple(expect):
                raise ValueError("device array must be contiguous")
        return DeviceArray(cai["shape"], dt, ptr=cai["data"][0], owner=x)
    return to_device(x, dtype, stream)


class PinnedArray:
    """Page-locked host array (for the end-to-end path): ``.array`` is a NumPy view."""

    def __init__(self, shape, dtype):
        self.shape = tuple(int(s) for s in (shape if isinstance(shape, (tuple, list)) else (shape,)))
        self.dtype = np.dtype(dtype)
        self.nbytes = int(np.prod(self.shape, dtype=np.int64)) * self.dtype.itemsize
        h = C.c_void_p()
        N.check(N.lib().ssdg_host_alloc(C.byref(h), max(self.nbytes, 1)), "host_alloc")
        self.ptr = h.value
        buf = (C.c_byte * max(self.nbytes, 1)).from_address(self.ptr)
        self.array = np.frombuffer(buf, dtype=self.dtype, count=self.size).reshape(self.shape)

    @property
    def size(self):
        return int(np.prod(self.shape, dtype=np.int64))

    def __del__(self):
        try:
            if self.ptr:
                self.array = None
                N.lib().ssdg_host_free(self.ptr)
                self.ptr = 0
        except Exception:
            pass
