"""ctypes binding of include/signalops.h — the same calls julia/GPUSink.jl makes
through `ccall`.  There is deliberately no fallback: if the shared library is
missing or no B200 is visible, every entry point raises."""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(os.path.dirname(_HERE), "lib", "libsignalops_cuda.so")

ABI_VERSION = 1
F32, F64, I64 = 1, 2, 3
SYMBOLS = ["sigops_abi_version", "sigops_device_count", "sigops_ctx_create", "sigops_ctx_destroy",
           "sigops_last_error", "sigops_plan_create", "sigops_plan_destroy", "sigops_plan_run",
           "sigops_plan_run_device", "sigops_plan_launch_count", "sigops_plan_algorithmic_bytes",
           "sigops_measure_peaks", "sigops_ctx_set_profiling", "sigops_profile_collect",
           "sigops_host_alloc", "sigops_host_free", "sigops_plan_run_ragged"]
KERNEL_KINDS = ["map", "iir_main", "iir_carry", "iir_fix", "fir"]


class Buffer(C.Structure):
    _fields_ = [("ptr", C.c_void_p), ("nframes", C.c_int64), ("nchannels", C.c_int32),
                ("dtype", C.c_int32), ("ld", C.c_int64)]


class Stats(C.Structure):
    _fields_ = [("gpu_ms", C.c_double), ("h2d_ms", C.c_double), ("d2h_ms", C.c_double),
                ("wall_ms", C.c_double), ("launches", C.c_int64), ("h2d_bytes", C.c_int64),
                ("d2h_bytes", C.c_int64), ("out_samples", C.c_int64)]

    def asdict(self):
        return {n: getattr(self, n) for n, _ in self._fields_}


class SigopsError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"libsignalops_cuda: {msg} (code {code})")
        self.code = code
        self.msg = msg


_lib = None


def load():
    """Load the shared library (built by `__graft_entry__.build()` / csrc/Makefile)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise FileNotFoundError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'`. "
            "The GPU sink has no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    vp, i64 = C.c_void_p, C.c_int64
    lib.sigops_abi_version.restype = C.c_int
    lib.sigops_device_count.argtypes = [C.POINTER(C.c_int)]
    lib.sigops_ctx_create.argtypes = [C.POINTER(C.c_int), C.c_int, C.POINTER(vp)]
    lib.sigops_ctx_destroy.argtypes = [vp]
    lib.sigops_ctx_destroy.restype = None
    lib.sigops_last_error.argtypes = [vp]
    lib.sigops_last_error.restype = C.c_char_p
    lib.sigops_plan_create.argtypes = [vp, C.c_char_p, C.c_size_t, C.POINTER(vp)]
    lib.sigops_plan_destroy.argtypes = [vp]
    lib.sigops_plan_destroy.restype = None
    lib.sigops_plan_run.argtypes = [vp, i64, C.POINTER(Buffer), C.POINTER(Buffer), C.POINTER(Stats)]
    lib.sigops_plan_run_ragged.argtypes = [vp, i64, C.POINTER(Buffer), C.POINTER(Buffer), C.POINTER(i64), C.POINTER(Stats)]
    lib.sigops_plan_run_device.argtypes = [vp, C.c_int, i64, C.POINTER(Buffer), C.POINTER(Buffer),
                                           vp, C.POINTER(Stats)]
    lib.sigops_plan_launch_count.argtypes = [vp, C.POINTER(i64)]
    lib.sigops_plan_algorithmic_bytes.argtypes = [vp, C.POINTER(i64)]
    lib.sigops_measure_peaks.argtypes = [vp, C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_double)]
    lib.sigops_ctx_set_profiling.argtypes = [vp, C.c_int]
    lib.sigops_profile_collect.argtypes = [vp, C.c_int, C.POINTER(C.c_double), C.POINTER(i64), C.c_int]
    lib.sigops_host_alloc.argtypes = [C.c_size_t, C.POINTER(vp)]
    lib.sigops_host_free.argtypes = [vp]
    if lib.sigops_abi_version() != ABI_VERSION:
        raise RuntimeError("libsignalops_cuda.so ABI version mismatch")
    _lib = lib
    return lib


def _check(lib, ctx, code):
    if code != 0:
        msg = lib.sigops_last_error(ctx)
        raise SigopsError(code, msg.decode("utf-8", "replace") if msg else "unknown error")


def dtype_code(dt):
    """Sample type code of a host buffer handed to the C ABI: exactly the three types the device
    reads and writes.  Anything else (Int32, Int16, ...) must be converted by the caller first —
    silently treating it as Int64 would read or write past the array."""
    dt = np.dtype(dt)
    if dt == np.float32:
        return F32
    if dt == np.float64:
        return F64
    if dt == np.int64:
        return I64
    raise TypeError(f"host buffers must be float32, float64 or int64, not {dt}")


_PIN_POOL = {}                 # rounded size -> free page-locked blocks (page-locking costs ~0.6 s per GB: reuse them)
_PIN_POOL_BYTES = 0
_PIN_POOL_CAP = 16 << 30


class _PinnedBlock:
    """Owner of one sigops_host_alloc block.  When the last array viewing it is collected the block goes back to a
    small pool (size-bucketed, capped) instead of being unlocked: a steady stream of `sink` results then never
    pays for page-locking again.  (The Julia glue does the same from the result array's finalizer.)"""

    def __init__(self, nbytes):
        global _PIN_POOL_BYTES
        self.lib = load()
        self.size = max((int(nbytes) + (1 << 20) - 1) >> 20 << 20, 1 << 20)
        free = _PIN_POOL.get(self.size)
        if free:
            self.ptr = C.c_void_p(free.pop())
            _PIN_POOL_BYTES -= self.size
        else:
            self.ptr = C.c_void_p()
            _check(self.lib, None, self.lib.sigops_host_alloc(self.size, C.byref(self.ptr)))
        self.nbytes = int(nbytes)

    def __del__(self):
        global _PIN_POOL_BYTES
        try:
            if self.ptr:
                if _PIN_POOL_BYTES + self.size <= _PIN_POOL_CAP:
                    _PIN_POOL.setdefault(self.size, []).append(self.ptr.value)
                    _PIN_POOL_BYTES += self.size
                else:
                    self.lib.sigops_host_free(self.ptr)
                self.ptr = C.c_void_p()
        except Exception:
            pass


def release_pinned_pool():
    """Unlock and free every pooled block."""
    global _PIN_POOL_BYTES
    lib = load()
    for free in _PIN_POOL.values():
        while free:
            lib.sigops_host_free(C.c_void_p(free.pop()))
    _PIN_POOL_BYTES = 0


def pinned_empty(shape, dtype, order="F"):
    """numpy array in page-locked memory (the result of `sink(x, GPUSink())` is allocated by the sink, so it
    can live where the DMA engines write directly — include/signalops.h `sigops_host_alloc`)."""
    dt = np.dtype(dtype)
    n = int(np.prod(shape)) if len(shape) else 1
    blk = _PinnedBlock(n * dt.itemsize)
    buf = (C.c_char * max(n * dt.itemsize, 1)).from_address(blk.ptr.value)
    buf._owner = blk                                   # keeps the block alive as long as any view of `buf` exists
    return np.frombuffer(buf, dtype=dt, count=n).reshape(shape, order=order)


class Context:
    def __init__(self, devices=None):
        self.lib = load()
        self.handle = C.c_void_p()
        devs = list(devices) if devices else [0]
        arr = (C.c_int * len(devs))(*devs)
        _check(self.lib, None, self.lib.sigops_ctx_create(arr, len(devs), C.byref(self.handle)))
        self.devices = devs

    def close(self):
        if self.handle:
            self.lib.sigops_ctx_destroy(self.handle)
            self.handle = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_profiling(self, on):
        _check(self.lib, self.handle, self.lib.sigops_ctx_set_profiling(self.handle, 1 if on else 0))

    def profile_collect(self, dev_index=0):
        """{kind: (total_ms, launches)} since profiling was enabled / last collected."""
        n = len(KERNEL_KINDS)
        ms = (C.c_double * n)()
        cnt = (C.c_int64 * n)()
        _check(self.lib, self.handle, self.lib.sigops_profile_collect(self.handle, dev_index, ms, cnt, n))
        return {k: (ms[i], cnt[i]) for i, k in enumerate(KERNEL_KINDS) if cnt[i]}

    def measure_peaks(self, dev_index=0):
        a, b = C.c_double(), C.c_double()
        _check(self.lib, self.handle, self.lib.sigops_measure_peaks(self.handle, dev_index, C.byref(a), C.byref(b)))
        return a.value, b.value


class CompiledPlan:
    def __init__(self, ctx: Context, plan_bytes: bytes):
        self.ctx = ctx
        self.lib = ctx.lib
        self.handle = C.c_void_p()
        _check(self.lib, ctx.handle, self.lib.sigops_plan_create(ctx.handle, plan_bytes, len(plan_bytes),
                                                               C.byref(self.handle)))

    def close(self):
        if self.handle:
            self.lib.sigops_plan_destroy(self.handle)
            self.handle = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @staticmethod
    def host_buffers(arrays):
        """arrays: list of Fortran-ordered or 1-D/2-D numpy arrays -> Buffer array.
        A (N,C) array must be column-major so each channel is contiguous in time
        (the Julia layout); C-ordered input is copied by the caller beforehand."""
        bufs = (Buffer * len(arrays))()
        for k, a in enumerate(arrays):
            if hasattr(a, "raw") and hasattr(a, "enc"):          # wav.WavRaw: frame-interleaved file layout
                n, c = a.raw.shape
                bufs[k] = Buffer(a.raw.ctypes.data, n, c, a.enc | 0x100, n)
                continue
            n, c = (a.shape[0], 1) if a.ndim == 1 else a.shape
            if a.ndim == 2 and c > 1 and n > 0 and (a.strides[1] < n * a.itemsize or a.strides[1] % a.itemsize):
                raise ValueError("multi-channel host buffers must be column-major (channels at least nframes apart)")
            if n > 1 and a.strides[0] != a.itemsize:
                raise ValueError("host buffers must be dense along time (stride of one element); "
                                 "copy strided views with numpy.ascontiguousarray first")
            ld = n if a.ndim == 1 or c == 1 else a.strides[1] // a.itemsize
            bufs[k] = Buffer(a.ctypes.data, n, c, dtype_code(a.dtype), max(ld, n))
        return bufs

    def run_host(self, ninst, in_arrays, out_arrays):
        ins = self.host_buffers(in_arrays)
        outs = self.host_buffers(out_arrays)
        st = Stats()
        _check(self.lib, self.ctx.handle, self.lib.sigops_plan_run(self.handle, ninst, ins, outs, C.byref(st)))
        return st.asdict()

    def run_ragged(self, ninst, in_arrays, out_arrays, temp_frames):
        """Instances of different lengths (include/signalops.h `sigops_plan_run_ragged`): each array holds the
        instance's own frames; `temp_frames` [ninst][n_temps] the valid frames of the plan's temps."""
        ins = self.host_buffers(in_arrays)
        outs = self.host_buffers(out_arrays)
        tf = np.ascontiguousarray(temp_frames, dtype=np.int64)
        st = Stats()
        _check(self.lib, self.ctx.handle, self.lib.sigops_plan_run_ragged(
            self.handle, ninst, ins, outs, tf.ctypes.data_as(C.POINTER(C.c_int64)), C.byref(st)))
        return st.asdict()

    def run_device(self, ninst, in_bufs, out_bufs, stream=None, dev_index=0, want_stats=False):
        """in_bufs/out_bufs: ctypes Buffer arrays holding device pointers."""
        st = Stats()
        _check(self.lib, self.ctx.handle, self.lib.sigops_plan_run_device(
            self.handle, dev_index, ninst, in_bufs, out_bufs, C.c_void_p(stream) if stream else None,
            C.byref(st) if want_stats else None))
        return st.asdict() if want_stats else None

    def launch_count(self):
        v = C.c_int64()
        _check(self.lib, self.ctx.handle, self.lib.sigops_plan_launch_count(self.handle, C.byref(v)))
        return v.value

    def algorithmic_bytes(self):
        v = C.c_int64()
        _check(self.lib, self.ctx.handle, self.lib.sigops_plan_algorithmic_bytes(self.handle, C.byref(v)))
        return v.value
