"""Zero-copy DLPack export of OkEnv device buffers (no compiled extension needed).

A ``DLManagedTensor`` is built with ctypes around the device pointer that ``ok_get_buffer`` returns and
wrapped in a ``PyCapsule`` named ``"dltensor"``; ``torch.from_dlpack`` (or any DLPack consumer) adopts it.
The capsule's deleter drops a reference on the owning :class:`~openkitchen_b200.env.Env`, so a tensor keeps
its env -- and therefore the memory -- alive.  Layout follows dlpack.h v0.8 (the ABI torch consumes).
"""
from __future__ import annotations

import atexit
import ctypes as C

import numpy as np

kDLCUDA = 2
kDLInt, kDLUInt, kDLFloat = 0, 1, 2


class DLDevice(C.Structure):
    _fields_ = [("device_type", C.c_int32), ("device_id", C.c_int32)]


class DLDataType(C.Structure):
    _fields_ = [("code", C.c_uint8), ("bits", C.c_uint8), ("lanes", C.c_uint16)]


class DLTensor(C.Structure):
    _fields_ = [
        ("data", C.c_void_p),
        ("device", DLDevice),
        ("ndim", C.c_int32),
        ("dtype", DLDataType),
        ("shape", C.POINTER(C.c_int64)),
        ("strides", C.POINTER(C.c_int64)),
        ("byte_offset", C.c_uint64),
    ]


class DLManagedTensor(C.Structure):
    pass


_DELETER = C.CFUNCTYPE(None, C.POINTER(DLManagedTensor))
DLManagedTensor._fields_ = [("dl_tensor", DLTensor), ("manager_ctx", C.c_void_p), ("deleter", _DELETER)]

_CODES = {np.dtype(np.float32): (kDLFloat, 32), np.dtype(np.int32): (kDLInt, 32), np.dtype(np.uint32): (kDLUInt, 32),
          np.dtype(np.uint8): (kDLUInt, 8)}

_live = {}  # id -> (managed tensor, shape array, owner): everything the consumer may still touch

C.pythonapi.PyCapsule_New.restype = C.py_object
C.pythonapi.PyCapsule_New.argtypes = [C.c_void_p, C.c_char_p, C.c_void_p]


def live_exports(owner) -> int:
    """DLPack tensors exported from `owner` that some consumer still holds"""
    return sum(1 for _m, _s, o in _live.values() if o is owner)


@_DELETER
def _release(managed_ptr):
    rec = _live.pop(C.addressof(managed_ptr.contents), None)
    if rec is not None:
        owner = rec[2]
        # an env whose close() arrived while tensors were still alive is destroyed with its last export
        if getattr(owner, "_close_pending", False) and live_exports(owner) == 0:
            owner._destroy_now()


@atexit.register
def _detach_at_exit():
    """Tensors that are still alive when the interpreter shuts down are released by their consumer AFTER Python is
    gone: calling back into ``_release`` then is a crash.  Clear their deleter (DLPack allows a NULL deleter) and leak
    the few bytes of descriptor they point to."""
    for m, shp, _owner in list(_live.values()):
        C.cast(C.byref(m, DLManagedTensor.deleter.offset), C.POINTER(C.c_void_p))[0] = None
        C.pythonapi.Py_IncRef(C.py_object(m))
        C.pythonapi.Py_IncRef(C.py_object(shp))


def to_capsule(ptr: int, shape, dtype, device_id: int, owner):
    """DLPack capsule over ``ptr`` (device memory on CUDA device ``device_id``), keeping ``owner`` alive."""
    code, bits = _CODES[np.dtype(dtype)]
    shp = (C.c_int64 * len(shape))(*shape)
    m = DLManagedTensor()
    m.dl_tensor.data = ptr
    m.dl_tensor.device = DLDevice(kDLCUDA, device_id)
    m.dl_tensor.ndim = len(shape)
    m.dl_tensor.dtype = DLDataType(code, bits, 1)
    m.dl_tensor.shape = shp
    m.dl_tensor.strides = None  # compact row-major
    m.dl_tensor.byte_offset = 0
    m.manager_ctx = None
    m.deleter = _release
    _live[C.addressof(m)] = (m, shp, owner)
    return C.pythonapi.PyCapsule_New(C.addressof(m), b"dltensor", None)


class DeviceBuffer:
    """``__dlpack__`` provider for one OkEnv buffer (what ``torch.from_dlpack`` expects)."""

    def __init__(self, env, name: str, info=None):
        """info: (device pointer, shape, dtype) of a device array the env owns that is not an OkBuffer (e.g. the
        reset-draw counters); None = env.buffer_info(name)"""
        self.env, self.name = env, name
        self.ptr, self.shape, self.dtype = info if info is not None else env.buffer_info(name)

    def __dlpack__(self, stream=None, **_):
        """`stream` (DLPack protocol: the consumer's stream; 1 = legacy default, 2 = per-thread default, -1 = no sync):
        the buffers are produced on torch's current stream of the env's device (where BatchEnv launches), so a consumer
        on another stream is made to wait for an event recorded there."""
        if stream is not None and stream != -1:
            try:
                import torch

                dev = int(self.env.cfg.device)
                cur = torch.cuda.current_stream(dev)
                target = 0 if stream in (0, 1) else int(stream)
                if stream != 2 and cur.cuda_stream != target:
                    ev = torch.cuda.Event()
                    ev.record(cur)
                    torch.cuda.ExternalStream(target, device=dev).wait_event(ev)
            except ImportError:
                pass
        return to_capsule(self.ptr, self.shape, self.dtype, int(self.env.cfg.device), self.env)

    def __dlpack_device__(self):
        return (kDLCUDA, int(self.env.cfg.device))

    @property
    def __cuda_array_interface__(self):
        return {"shape": tuple(self.shape), "typestr": np.dtype(self.dtype).str, "data": (self.ptr, False), "version": 3,
                "strides": None}
