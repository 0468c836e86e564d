"""neo_b200 -- host-side Python mirror of the reference's front end over the C ABI (include/neo_b200.h).

The reference's Python package is a thin pybind11 layer (extra/python/src/main.cpp:130-198, extra/python/src/neo/fft/__init__.py:20-29):
``neo.fft.fft(x, n, norm)``, ``neo.fft.ifft``, ``neo.convolve(in1, in2, mode, method)``. The same names live here, plus the plan /
convolver objects the C++ drivers use (Plan(order) + call on spans; Convolver.filter(H) + call on a block), batched.

Everything computes on the GPU through ``libneo_b200.so``. There is NO CPU fallback: if the library is missing or no CUDA
device is usable, importing works but every compute call raises ``RuntimeError``.

numpy arrays are HOST buffers (copied to the device and back inside the call, synchronous like the reference);
objects with ``data_ptr()`` / ``__cuda_array_interface__`` (torch CUDA tensors) are DEVICE buffers used in place, the work
is enqueued on the handle's stream.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Any

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
# NEO_B200_LIBRARY: another build of the same library (A/B measurements of compile-time choices); never a fallback
LIBRARY_PATH = os.environ.get("NEO_B200_LIBRARY") or os.path.join(_HERE, "libneo_b200.so")

F32, F64 = 0, 1
FORWARD, BACKWARD = -1, 1
HOST, DEVICE = 0, 1
UPOLS, UPOLA = 0, 1
DIAGONAL, MATRIX = 0, 1

_vp, _sz, _i = C.c_void_p, C.c_size_t, C.c_int


class ConvConfig(C.Structure):
    _fields_ = [
        ("kind", _i),
        ("dtype", _i),
        ("topology", _i),
        ("outputs", _sz),
        ("inputs", _sz),
        ("block", _sz),
        ("partitions", _sz),
        ("max_blocks", _sz),
        ("partition_begin", _sz),
        ("partition_end", _sz),
        ("frame_blocks", _sz),
        ("input_delayed", _sz),
    ]


class BankLayout(C.Structure):
    _fields_ = [("channel_groups", _sz), ("partition_shards", _sz)]


class BankRankInfo(C.Structure):
    _fields_ = [
        ("rank", _i),
        ("device", _i),
        ("channel_group", _sz),
        ("partition_shard", _sz),
        ("group_first", _sz),
        ("group_count", _sz),
        ("in_first", _sz),
        ("in_count", _sz),
        ("out_first", _sz),
        ("out_count", _sz),
        ("partition_begin", _sz),
        ("partition_end", _sz),
        ("delay_blocks", _sz),
    ]


class LowLatConfig(C.Structure):
    _fields_ = [
        ("dtype", _i),
        ("channels", _sz),
        ("block", _sz),
        ("partitions", _sz),
        ("levels", _sz),
        ("frame_blocks", _sz * 4),
    ]


BANK_ID_BYTES = 128
_pp = C.POINTER(_vp)

# name -> (restype, argtypes): exactly the entry points include/neo_b200.h declares
SIGNATURES = {
    "neo_b200_last_error": (C.c_char_p, []),
    "neo_b200_version": (C.c_char_p, []),
    "neo_b200_device_count": (_i, []),
    "neo_b200_set_device": (_i, [_i]),
    "neo_b200_kernel_launches": (_i, [C.POINTER(C.c_uint64)]),
    "neo_b200_fft_plan_create": (_i, [C.POINTER(_vp), _sz, _i]),
    "neo_b200_fft_plan_destroy": (None, [_vp]),
    "neo_b200_fft_plan_order": (_sz, [_vp]),
    "neo_b200_fft_plan_size": (_sz, [_vp]),
    "neo_b200_fft_max_order": (_sz, []),
    "neo_b200_fft_exec": (_i, [_vp, _vp, _vp, _sz, _i, _i]),
    "neo_b200_fft_exec_split": (_i, [_vp, _vp, _vp, _vp, _vp, _sz, _i, _i]),
    "neo_b200_fft_exec_strided": (_i, [_vp, _vp, C.c_ssize_t, _vp, C.c_ssize_t, _i]),
    "neo_b200_fft_plan_set_stream": (_i, [_vp, _vp]),
    "neo_b200_fft_plan_synchronize": (_i, [_vp]),
    "neo_b200_fft_convolver_create": (_i, [C.POINTER(_vp), _sz, _sz, _i]),
    "neo_b200_fft_convolver_destroy": (None, [_vp]),
    "neo_b200_fft_convolver_output_size": (_sz, [_vp]),
    "neo_b200_fft_convolver_exec": (_i, [_vp, _vp, _vp, _vp, _sz, _i]),
    "neo_b200_num_stft_frames": (_sz, [_sz, _sz, _sz]),
    "neo_b200_stft": (_i, [_vp, _sz, _sz, _sz, _sz, _sz, _vp, _vp, _i, _i]),
    "neo_b200_dct2_plan_create": (_i, [C.POINTER(_vp), _sz, _i]),
    "neo_b200_dct2_plan_destroy": (None, [_vp]),
    "neo_b200_dct2_plan_order": (_sz, [_vp]),
    "neo_b200_dct2_plan_size": (_sz, [_vp]),
    "neo_b200_dct2_exec": (_i, [_vp, _vp, _vp, _sz, _i]),
    "neo_b200_dct2_plan_set_stream": (_i, [_vp, _vp]),
    "neo_b200_dft_plan_create": (_i, [C.POINTER(_vp), _sz, _i]),
    "neo_b200_dft_plan_destroy": (None, [_vp]),
    "neo_b200_dft_plan_size": (_sz, [_vp]),
    "neo_b200_dft_exec": (_i, [_vp, _vp, _vp, _sz, _i, _i]),
    "neo_b200_dft_plan_set_stream": (_i, [_vp, _vp]),
    "neo_b200_rfft_plan_create": (_i, [C.POINTER(_vp), _sz, _i]),
    "neo_b200_rfft_plan_destroy": (None, [_vp]),
    "neo_b200_rfft_plan_order": (_sz, [_vp]),
    "neo_b200_rfft_plan_size": (_sz, [_vp]),
    "neo_b200_rfft_exec": (_i, [_vp, _vp, _vp, _sz, _i]),
    "neo_b200_irfft_exec": (_i, [_vp, _vp, _sz, _vp, _sz, _i]),
    "neo_b200_rfft_plan_set_stream": (_i, [_vp, _vp]),
    "neo_b200_rfft_plan_synchronize": (_i, [_vp]),
    "neo_b200_bitrev_table": (_i, [_sz, _vp]),
    "neo_b200_digitrev_perm": (_i, [_sz, _sz, _vp]),
    "neo_b200_fdl_index_sequence": (_i, [_sz, _sz, _vp, _vp]),
    "neo_b200_num_partitions": (_sz, [_sz, _sz]),
    "neo_b200_next_order": (_sz, [_sz]),
    "neo_b200_normalize_impulse": (_i, [_vp, _sz, _sz, _i, _i]),
    "neo_b200_uniform_partition": (_i, [_vp, _sz, _sz, _sz, _vp, _i, _i]),
    "neo_b200_conv_create": (_i, [C.POINTER(_vp), C.POINTER(ConvConfig)]),
    "neo_b200_conv_destroy": (None, [_vp]),
    "neo_b200_conv_set_filter": (_i, [_vp, _vp, _i]),
    "neo_b200_conv_set_filter_csr": (_i, [_vp, _vp, _vp, _vp, _vp]),
    "neo_b200_compressed_fdl_create": (_i, [C.POINTER(_vp), _sz, _sz, _i, _i]),
    "neo_b200_compressed_fdl_destroy": (None, [_vp]),
    "neo_b200_compressed_fdl_insert": (_i, [_vp, _vp, _sz, _i]),
    "neo_b200_compressed_fdl_row": (_i, [_vp, _sz, _vp, _i]),
    "neo_b200_compressed_fdl_raw": (_i, [_vp, _sz, _vp]),
    "neo_b200_conv_set_impulse": (_i, [_vp, _vp, _sz, _i]),
    "neo_b200_conv_stage_filter": (_i, [_vp, _vp, _i]),
    "neo_b200_conv_stage_impulse": (_i, [_vp, _vp, _sz, _i]),
    "neo_b200_conv_crossfade": (_i, [_vp, _sz, _sz, C.POINTER(_sz)]),
    "neo_b200_conv_reset": (_i, [_vp]),
    "neo_b200_conv_process": (_i, [_vp, _vp, _vp, _sz, _i]),
    "neo_b200_conv_forward": (_i, [_vp, _vp, _sz, _i]),
    "neo_b200_conv_forward_range": (_i, [_vp, _vp, _sz, _sz, _sz, _i]),
    "neo_b200_conv_spectra": (_i, [_vp, C.POINTER(_vp), C.POINTER(_sz)]),
    "neo_b200_conv_inverse": (_i, [_vp, _vp, _vp, _sz, _sz, _sz, _i]),
    "neo_b200_conv_process_window": (_i, [_vp, _vp, _vp, _i, _i]),
    "neo_b200_conv_tail": (_i, [_vp, _vp, _i]),
    "neo_b200_conv_set_stream": (_i, [_vp, _vp]),
    "neo_b200_conv_synchronize": (_i, [_vp]),
    "neo_b200_conv_profile_enable": (_i, [_vp, _i]),
    "neo_b200_conv_profile_read": (_i, [_vp, C.POINTER(C.c_double), C.POINTER(C.c_uint64)]),
    "neo_b200_conv_device_bytes": (_sz, [_vp]),
    "neo_b200_lowlat_layout": (_i, [C.POINTER(LowLatConfig), C.POINTER(_sz), C.POINTER(_sz), C.POINTER(_sz)]),
    "neo_b200_lowlat_create": (_i, [C.POINTER(_vp), C.POINTER(LowLatConfig)]),
    "neo_b200_lowlat_destroy": (None, [_vp]),
    "neo_b200_lowlat_set_filter": (_i, [_vp, _vp, _i]),
    "neo_b200_lowlat_set_impulse": (_i, [_vp, _vp, _sz, _i]),
    "neo_b200_lowlat_reset": (_i, [_vp]),
    "neo_b200_lowlat_process": (_i, [_vp, _vp, _vp, _sz, _i]),
    "neo_b200_lowlat_process_samples": (_i, [_vp, _vp, _vp, _sz, _i]),
    "neo_b200_lowlat_stage_filter": (_i, [_vp, _vp, _i]),
    "neo_b200_lowlat_stage_impulse": (_i, [_vp, _vp, _sz, _i]),
    "neo_b200_lowlat_crossfade": (_i, [_vp, _sz, C.POINTER(_sz)]),
    "neo_b200_lowlat_set_stream": (_i, [_vp, _vp]),
    "neo_b200_lowlat_synchronize": (_i, [_vp]),
    "neo_b200_lowlat_device_bytes": (_sz, [_vp]),
    "neo_b200_bank_unique_id": (_i, [_vp]),
    "neo_b200_bank_create": (_i, [C.POINTER(_vp), C.POINTER(ConvConfig), C.POINTER(BankLayout), C.POINTER(_i), _sz]),
    "neo_b200_bank_create_rank": (_i, [C.POINTER(_vp), C.POINTER(ConvConfig), C.POINTER(BankLayout), _i, _i, _i, _vp]),
    "neo_b200_bank_destroy": (None, [_vp]),
    "neo_b200_bank_local_ranks": (_i, [_vp, C.POINTER(_sz)]),
    "neo_b200_bank_local_rank": (_i, [_vp, _sz, C.POINTER(BankRankInfo)]),
    "neo_b200_bank_layout_info": (_i, [C.POINTER(ConvConfig), C.POINTER(BankLayout), _sz, C.POINTER(BankRankInfo)]),
    "neo_b200_bank_set_impulse": (_i, [_vp, _pp, _sz, _i]),
    "neo_b200_bank_set_filter": (_i, [_vp, _pp, _i]),
    "neo_b200_bank_reset": (_i, [_vp]),
    "neo_b200_bank_submit": (_i, [_vp, _pp, _pp, _sz, _i]),
    "neo_b200_bank_wait": (_i, [_vp]),
    "neo_b200_bank_process": (_i, [_vp, _pp, _pp, _sz, _i]),
    "neo_b200_bank_timer_start": (_i, [_vp]),
    "neo_b200_bank_timer_stop": (_i, [_vp, C.POINTER(C.c_double)]),
    "neo_b200_bank_profile_enable": (_i, [_vp, _i]),
    "neo_b200_bank_profile_read": (_i, [_vp, _sz, C.POINTER(C.c_double), C.POINTER(C.c_uint64)]),
    "neo_b200_bank_device_bytes": (_sz, [_vp, _sz]),
}

_lib = None


def library() -> C.CDLL:
    """The C-ABI library; raises if it has not been built (no fallback of any kind)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIBRARY_PATH):
            raise RuntimeError(
                f"{LIBRARY_PATH} is missing: build it with `make -C neo-dsp_b200` (or __graft_entry__.build()); "
                "neo_b200 has no CPU fallback"
            )
        lib = C.CDLL(LIBRARY_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype, fn.argtypes = res, args
        _lib = lib
    return _lib


def _check(status: int) -> None:
    if status != 0:
        raise RuntimeError(library().neo_b200_last_error().decode())


def kernel_launches() -> int:
    n = C.c_uint64(0)
    _check(library().neo_b200_kernel_launches(C.byref(n)))
    return int(n.value)


def device_count() -> int:
    return int(library().neo_b200_device_count())


def set_device(index: int) -> None:
    _check(library().neo_b200_set_device(index))


# ---- buffers ---------------------------------------------------------------------------------------------------------
_REAL_OF = {"complex64": "float32", "complex128": "float64", "float32": "float32", "float64": "float64"}
_DTYPE_CODE = {"float32": F32, "float64": F64}


def _is_device(a: Any) -> bool:
    return hasattr(a, "data_ptr") and getattr(a, "is_cuda", False)


def _dtype_name(a: Any) -> str:
    return str(a.dtype).replace("torch.", "")


def _ptr(a: Any) -> int:
    if _is_device(a):
        if not a.is_contiguous():
            raise ValueError("device buffers must be contiguous")
        return int(a.data_ptr())
    if not isinstance(a, np.ndarray) or not a.flags.c_contiguous:
        raise ValueError("host buffers must be C-contiguous numpy arrays")
    return int(a.ctypes.data)


def _space(a: Any) -> int:
    return DEVICE if _is_device(a) else HOST


def _empty_like_kind(a: Any, shape, dtype_name: str):
    if _is_device(a):
        import torch

        return torch.empty(shape, dtype=getattr(torch, dtype_name), device=a.device)
    return np.empty(shape, dtype=dtype_name)


def _stream_ptr(stream: Any) -> int:
    return int(getattr(stream, "cuda_stream", stream) or 0)


# ---- plans -----------------------------------------------------------------------------------------------------------
class FFTPlan:
    """neo::fft::fft_plan<Complex>{from_order, order} (fft/reference/c2c_dit2_plan.hpp:22-104), batched over leading axes."""

    def __init__(self, order: int, dtype="complex64"):
        self.real = _REAL_OF[str(np.dtype(dtype))]
        self.complex = "complex64" if self.real == "float32" else "complex128"
        self._h = _vp()
        _check(library().neo_b200_fft_plan_create(C.byref(self._h), order, _DTYPE_CODE[self.real]))

    @staticmethod
    def max_order() -> int:
        return int(library().neo_b200_fft_max_order())

    @staticmethod
    def max_size() -> int:
        return 1 << FFTPlan.max_order()

    def order(self) -> int:
        return int(library().neo_b200_fft_plan_order(self._h))

    def size(self) -> int:
        return int(library().neo_b200_fft_plan_size(self._h))

    def set_stream(self, stream) -> None:
        _check(library().neo_b200_fft_plan_set_stream(self._h, _stream_ptr(stream)))

    def synchronize(self) -> None:
        _check(library().neo_b200_fft_plan_synchronize(self._h))

    def __call__(self, x, direction: int = FORWARD, out=None):
        """plan(x, dir): in place when `out` is None (like the reference), else out-of-place. x[..., size]."""
        if _dtype_name(x) != self.complex or x.shape[-1] != self.size():
            raise ValueError(f"expected {self.complex}[..., {self.size()}]")
        out = x if out is None else out
        batch = int(np.prod(x.shape[:-1], dtype=np.int64)) if x.ndim > 1 else 1
        _check(library().neo_b200_fft_exec(self._h, _ptr(x), _ptr(out), batch, direction, _space(x)))
        return out

    def split(self, re, im, direction: int = FORWARD):
        """neo::fft::split_fft_plan (fft/fallback/fallback_split_fft_plan.hpp:27-51): in-place transform of separate real and
        imaginary planes re[..., size], im[..., size]."""
        if _dtype_name(re) != self.real or _dtype_name(im) != self.real or re.shape != im.shape or re.shape[-1] != self.size():
            raise ValueError(f"expected two {self.real}[..., {self.size()}] planes")
        batch = int(np.prod(re.shape[:-1], dtype=np.int64)) if re.ndim > 1 else 1
        _check(library().neo_b200_fft_exec_split(self._h, _ptr(re), _ptr(im), _ptr(re), _ptr(im), batch, direction, _space(re)))
        return re, im

    def strided(self, x: np.ndarray, direction: int = FORWARD) -> None:
        """In-place transform of a strided rank-1 numpy view (layout_stride mdspan, fft_test.cpp:114-128)."""
        if x.ndim != 1 or x.shape[0] != self.size() or str(x.dtype) != self.complex:
            raise ValueError("expected a rank-1 complex view of plan size")
        stride = x.strides[0] // x.itemsize
        _check(library().neo_b200_fft_exec_strided(self._h, x.ctypes.data, stride, x.ctypes.data, stride, direction))

    def close(self) -> None:
        if self._h:
            library().neo_b200_fft_plan_destroy(self._h)
            self._h = _vp()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class DCT2Plan:
    """neo::fft::fallback_dct2_plan<Float>{from_order, order} (fft/dct.hpp:24-68): unnormalised type-2 DCT, batched over leading axes."""

    def __init__(self, order: int, dtype="float32"):
        self.real = _REAL_OF[str(np.dtype(dtype))]
        self._h = _vp()
        _check(library().neo_b200_dct2_plan_create(C.byref(self._h), order, _DTYPE_CODE[self.real]))

    def order(self) -> int:
        return int(library().neo_b200_dct2_plan_order(self._h))

    def size(self) -> int:
        return int(library().neo_b200_dct2_plan_size(self._h))

    def set_stream(self, stream) -> None:
        _check(library().neo_b200_dct2_plan_set_stream(self._h, _stream_ptr(stream)))

    def __call__(self, x, out=None):
        """plan(x): in place when `out` is None (like the reference). x[..., size] reals."""
        if _dtype_name(x) != self.real or x.shape[-1] != self.size():
            raise ValueError(f"expected {self.real}[..., {self.size()}]")
        out = x if out is None else out
        batch = int(np.prod(x.shape[:-1], dtype=np.int64)) if x.ndim > 1 else 1
        _check(library().neo_b200_dct2_exec(self._h, _ptr(x), _ptr(out), batch, _space(x)))
        return out

    def close(self) -> None:
        if self._h:
            library().neo_b200_dct2_plan_destroy(self._h)
            self._h = _vp()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class DFTPlan:
    """neo::fft::dft_plan<Complex>{size} == fallback_dft_plan (fft/fallback/fallback_dft_plan.hpp:24-96): complex transform of ANY
    size through Bluestein's chirp-z, batched over leading axes, unnormalised both ways."""

    def __init__(self, size: int, dtype="complex64"):
        self.real = _REAL_OF[str(np.dtype(dtype))]
        self.complex = "complex64" if self.real == "float32" else "complex128"
        self._h = _vp()
        _check(library().neo_b200_dft_plan_create(C.byref(self._h), size, _DTYPE_CODE[self.real]))

    def size(self) -> int:
        return int(library().neo_b200_dft_plan_size(self._h))

    def set_stream(self, stream) -> None:
        _check(library().neo_b200_dft_plan_set_stream(self._h, _stream_ptr(stream)))

    def __call__(self, x, direction: int = FORWARD, out=None):
        """plan(x, dir): in place when `out` is None (like the reference), else out-of-place. x[..., size]."""
        if _dtype_name(x) != self.complex or x.shape[-1] != self.size():
            raise ValueError(f"expected {self.complex}[..., {self.size()}]")
        out = x if out is None else out
        batch = int(np.prod(x.shape[:-1], dtype=np.int64)) if x.ndim > 1 else 1
        _check(library().neo_b200_dft_exec(self._h, _ptr(x), _ptr(out), batch, direction, _space(x)))
        return out

    def close(self) -> None:
        if self._h:
            library().neo_b200_dft_plan_destroy(self._h)
            self._h = _vp()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class RFFTPlan:
    """neo::fft::rfft_plan<Float>{from_order, order} (fft/fallback/fallback_rfft_plan.hpp:15-61), batched."""

    def __init__(self, order: int, dtype="float32"):
        self.real = _REAL_OF[str(np.dtype(dtype))]
        self.complex = "complex64" if self.real == "float32" else "complex128"
        self._h = _vp()
        _check(library().neo_b200_rfft_plan_create(C.byref(self._h), order, _DTYPE_CODE[self.real]))

    def order(self) -> int:
        return int(library().neo_b200_rfft_plan_order(self._h))

    def size(self) -> int:
        return int(library().neo_b200_rfft_plan_size(self._h))

    def set_stream(self, stream) -> None:
        _check(library().neo_b200_rfft_plan_set_stream(self._h, _stream_ptr(stream)))

    def synchronize(self) -> None:
        _check(library().neo_b200_rfft_plan_synchronize(self._h))

    def rfft(self, x, out=None):
        """x[..., N] real -> [..., N/2+1] complex."""
        n = self.size()
        if _dtype_name(x) != self.real or x.shape[-1] != n:
            raise ValueError(f"expected {self.real}[..., {n}]")
        if out is None:
            out = _empty_like_kind(x, tuple(x.shape[:-1]) + (n // 2 + 1,), self.complex)
        batch = int(np.prod(x.shape[:-1], dtype=np.int64)) if x.ndim > 1 else 1
        _check(library().neo_b200_rfft_exec(self._h, _ptr(x), _ptr(out), batch, _space(x)))
        return out

    def irfft(self, x, out=None):
        """x[..., >= N/2+1] complex -> [..., N] real, UNNORMALISED (fallback_rfft_plan.hpp:39-55)."""
        n = self.size()
        if _dtype_name(x) != self.complex or x.shape[-1] < n // 2 + 1:
            raise ValueError(f"expected {self.complex}[..., >= {n // 2 + 1}]")
        if out is None:
            out = _empty_like_kind(x, tuple(x.shape[:-1]) + (n,), self.real)
        batch = int(np.prod(x.shape[:-1], dtype=np.int64)) if x.ndim > 1 else 1
        _check(library().neo_b200_irfft_exec(self._h, _ptr(x), x.shape[-1], _ptr(out), batch, _space(x)))
        return out

    def close(self) -> None:
        if self._h:
            library().neo_b200_rfft_plan_destroy(self._h)
            self._h = _vp()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


# ---- index tables (bit-exact contract) ----------------------------------------------------------------------------------
def bitrev_table(order: int) -> np.ndarray:
    out = np.zeros(1 << order, dtype=np.uint32)
    _check(library().neo_b200_bitrev_table(order, out.ctypes.data))
    return out


def digitrev_perm(radix: int, size: int) -> np.ndarray:
    out = np.zeros(size, dtype=np.uint32)
    _check(library().neo_b200_digitrev_perm(radix, size, out.ctypes.data))
    return out


def fdl_index_sequence(parts: int, calls: int):
    wp = np.zeros(calls, dtype=np.uint32)
    pairs = np.zeros((calls, parts, 2), dtype=np.uint32)
    _check(library().neo_b200_fdl_index_sequence(parts, calls, wp.ctypes.data, pairs.ctypes.data))
    return wp, pairs


def num_partitions(taps: int, block: int) -> int:
    return int(library().neo_b200_num_partitions(taps, block))


def next_order(size: int) -> int:
    return int(library().neo_b200_next_order(size))


# ---- filter preparation + convolver bank -----------------------------------------------------------------------------------
def uniform_partition(ir, block: int):
    """neo::convolution::uniform_partition (convolution/uniform_partition.hpp:13-26): ir[C][L] -> H[C][P][block+1]."""
    if ir.ndim != 2:
        raise ValueError("impulse response must be [channels][taps]")
    real = _dtype_name(ir)
    ch, taps = int(ir.shape[0]), int(ir.shape[1])
    parts = num_partitions(taps, block)
    out = _empty_like_kind(ir, (ch, parts, block + 1), "complex64" if real == "float32" else "complex128")
    _check(library().neo_b200_uniform_partition(_ptr(ir), ch, taps, block, _ptr(out), _DTYPE_CODE[real], _space(ir)))
    return out


def window(kind: str, size: int, dtype="float32") -> np.ndarray:
    """math/windowing.hpp:14-67: "rectangular", "hann" (the stft default) or "hamming" of `size` points, evaluated in `dtype`."""
    real = np.dtype(dtype).type
    if kind == "rectangular":
        return np.ones(size, dtype=real)
    i = np.arange(size, dtype=real)
    c = np.cos((real(np.pi) * real(2)) * i / real(size - 1)).astype(real)
    if kind == "hann":
        return (real(0.5) * (real(1) - c)).astype(real)
    if kind == "hamming":
        return (real(0.54) - real(0.46) * c).astype(real)
    raise ValueError(f"unknown window '{kind}'")


def num_stft_frames(signal: int, frame_size: int, overlap_size: int) -> int:
    return int(library().neo_b200_num_stft_frames(signal, frame_size, overlap_size))


def stft(x, frame_size: int, transform_size: int | None = None, overlap_size: int | None = None, window_kind="hann"):
    """neo::fft::stft(x, options) (fft/stft.hpp:39-125): x[C][L] reals -> [C][frames][bins] complex. Defaults follow
    stft_plan(transform_size) (:43-49): frame = transform, overlap = transform / 2, hann window. `window_kind` may also be an array
    of bit_ceil(transform_size) values."""
    if x.ndim != 2:
        raise ValueError("signal must be [channels][samples]")
    real = _dtype_name(x)
    transform_size = frame_size if transform_size is None else transform_size
    overlap_size = transform_size // 2 if overlap_size is None else overlap_size
    n = 1 << max(0, int(transform_size - 1).bit_length())
    ch, length = int(x.shape[0]), int(x.shape[1])
    frames = num_stft_frames(length, frame_size, overlap_size)
    out = _empty_like_kind(x, (ch, frames, n // 2 + 1), "complex64" if real == "float32" else "complex128")
    win = window(window_kind, n, real) if isinstance(window_kind, str) else window_kind
    wptr = None
    if not (isinstance(window_kind, str) and window_kind == "rectangular"):
        if _space(x) == DEVICE and isinstance(win, np.ndarray):
            import torch

            win = torch.from_numpy(np.ascontiguousarray(win)).to(x.device)
        wptr = _ptr(win)
    _check(library().neo_b200_stft(_ptr(x), ch, length, frame_size, transform_size, overlap_size, wptr, _ptr(out), _DTYPE_CODE[real], _space(x)))
    return out


def normalize_impulse(ir):
    """neo::convolution::normalize_impulse (convolution/normalize_impulse.hpp:13-33), in place on ir[C][L]; returns ir."""
    if ir.ndim != 2:
        raise ValueError("impulse response must be [channels][taps]")
    _check(library().neo_b200_normalize_impulse(_ptr(ir), int(ir.shape[0]), int(ir.shape[1]), _DTYPE_CODE[_dtype_name(ir)], _space(ir)))
    return ir


class CompressedFDL:
    """neo::convolution::compressed_fdl<FloatComplex, IntComplex> (compressed_fdl.hpp:17-52) on the device: `rows` rows of `cols`
    complex bins stored as int8 / int16 complex. insert(row, index) / row(index) (= operator[]) / raw(index) (the stored integers)."""

    def __init__(self, rows: int, cols: int, dtype="float32", bits: int = 16):
        self.real = np.dtype(dtype).name
        self.rows, self.cols, self.bits = int(rows), int(cols), int(bits)
        self._h = _vp()
        _check(library().neo_b200_compressed_fdl_create(C.byref(self._h), self.rows, self.cols, _DTYPE_CODE[self.real], self.bits))

    def insert(self, row, index: int) -> None:
        want = "complex64" if self.real == "float32" else "complex128"
        if _dtype_name(row) != want or int(row.shape[-1]) != self.cols:
            raise ValueError("row shape/dtype mismatch")
        _check(library().neo_b200_compressed_fdl_insert(self._h, _ptr(row), int(index), _space(row)))

    def row(self, index: int) -> np.ndarray:
        out = np.zeros(self.cols, dtype=np.complex64 if self.real == "float32" else np.complex128)
        _check(library().neo_b200_compressed_fdl_row(self._h, int(index), _ptr(out), HOST))
        return out

    def raw(self, index: int) -> np.ndarray:
        out = np.zeros((self.cols, 2), dtype=np.int8 if self.bits == 8 else np.int16)
        _check(library().neo_b200_compressed_fdl_raw(self._h, int(index), _ptr(out)))
        return out

    def close(self) -> None:
        if self._h:
            library().neo_b200_compressed_fdl_destroy(self._h)
            self._h = _vp()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Convolver:
    """A bank of neo::convolution::upols_convolver / upola_convolver instances
    (convolution/uniform_partitioned_convolver.hpp:14-65): `filter(H)` then call on blocks.

    H: DIAGONAL [C][P][B+1] (channel c has its own filter), MATRIX [O][I][P][B+1]. `stage_filter(H)` / `stage_impulse(ir)` then
    `crossfade(fade, delay)` switch to a new response mid-stream with a linear crossfade, keeping the delay line (overlap-save).
    """

    def __init__(self, kind: int = UPOLS, dtype="float32", topology: int = DIAGONAL, max_blocks: int = 1,
                 partition_range: tuple[int, int] | None = None, frame_blocks: int = 0):
        # frame_blocks = T > 0: every call carries exactly T blocks and the sum over partitions is evaluated by a second
        # overlap-save level along block time (neo_b200.h: neo_b200_conv_config::frame_blocks)
        self.kind, self.topology, self.max_blocks = kind, topology, (frame_blocks or max_blocks)
        self.frame_blocks = frame_blocks
        self.real = _REAL_OF[str(np.dtype(dtype))]
        self.partition_range = partition_range
        self._h = _vp()
        self.cfg = None
        self._stream = None

    def _create(self, outputs, inputs, block, partitions):
        self.close()
        self._spectra_view = None
        lo, hi = self.partition_range or (0, 0)
        self.cfg = ConvConfig(self.kind, _DTYPE_CODE[self.real], self.topology, outputs, inputs, block, partitions,
                              self.max_blocks, lo, hi, self.frame_blocks)
        _check(library().neo_b200_conv_create(C.byref(self._h), C.byref(self.cfg)))
        if self._stream is not None:
            _check(library().neo_b200_conv_set_stream(self._h, self._stream))

    def filter(self, H) -> None:
        """convolver.filter(partitions) (uniform_partitioned_convolver.hpp:38-45): deep copy, state zeroed."""
        want = 3 if self.topology == DIAGONAL else 4
        if H.ndim != want:
            raise ValueError(f"filter must have {want} dimensions for this topology")
        if _dtype_name(H) != ("complex64" if self.real == "float32" else "complex128"):
            raise ValueError("filter dtype does not match the convolver")
        outputs = int(H.shape[0])
        inputs = outputs if self.topology == DIAGONAL else int(H.shape[1])
        partitions, bins = int(H.shape[-2]), int(H.shape[-1])
        self._create(outputs, inputs, bins - 1, partitions)
        _check(library().neo_b200_conv_set_filter(self._h, _ptr(H), _space(H)))

    def filter_sparse(self, H, keep) -> None:
        """sparse convolvers' filter(partitions, sparsity) (sparse_filter.hpp:25-28): H [C][P][B+1] numpy, `keep` a boolean array of
        the same shape (the sparsity predicate evaluated per element). The CSR matrices are built here exactly as neo::csr_matrix
        builds them (row-major stored elements, csr_matrix.hpp:64-98) and handed to neo_b200_conv_set_filter_csr; the device keeps
        only the stored elements."""
        import numpy as np

        if self.topology != DIAGONAL or H.ndim != 3:
            raise ValueError("sparse filters: diagonal topology, H[C][P][B+1]")
        H = np.ascontiguousarray(H)
        keep = np.ascontiguousarray(keep, dtype=bool)
        if keep.shape != H.shape or _dtype_name(H) != ("complex64" if self.real == "float32" else "complex128"):
            raise ValueError("sparsity mask / dtype mismatch")
        outputs, partitions, bins = (int(v) for v in H.shape)
        self._create(outputs, outputs, bins - 1, partitions)
        counts = keep.sum(axis=2).astype(np.uint64)                       # [C][P] stored elements per row
        row_ptr = np.zeros((outputs, partitions + 1), dtype=np.uint64)
        row_ptr[:, 1:] = np.cumsum(counts, axis=1)
        base = np.zeros(outputs + 1, dtype=np.uint64)
        base[1:] = np.cumsum(row_ptr[:, -1])
        cols = np.ascontiguousarray(np.nonzero(keep)[2].astype(np.uint64))  # row-major order = CSR order
        vals = np.ascontiguousarray(H[keep])
        self.csr = (row_ptr, cols, vals, base)
        _check(library().neo_b200_conv_set_filter_csr(self._h, _ptr(vals) if vals.size else None, _ptr(cols) if cols.size else _ptr(base),
                                                      _ptr(row_ptr), _ptr(base)))

    def impulse(self, ir, block: int) -> None:
        """filter(uniform_partition(ir, block)) without materialising H on the host. ir: [C][L] or [O][I][L]."""
        want = 2 if self.topology == DIAGONAL else 3
        if ir.ndim != want or _dtype_name(ir) != self.real:
            raise ValueError("impulse response shape/dtype mismatch")
        outputs = int(ir.shape[0])
        inputs = outputs if self.topology == DIAGONAL else int(ir.shape[1])
        taps = int(ir.shape[-1])
        self._create(outputs, inputs, block, num_partitions(taps, block))
        _check(library().neo_b200_conv_set_impulse(self._h, _ptr(ir), taps, _space(ir)))

    def stage_filter(self, H) -> None:
        """H of this handle's shape ([C][P][B+1] diagonal, [O][I][P][B+1] matrix), prepared next to the current filter for
        `crossfade`: no output, delay line or sample count changes (neo_b200_conv_stage_filter)."""
        if self.cfg is None:
            raise RuntimeError("no filter set")
        lead = (int(self.cfg.outputs),) if self.topology == DIAGONAL else (int(self.cfg.outputs), int(self.cfg.inputs))
        shape = lead + (int(self.cfg.partitions), int(self.cfg.block) + 1)
        if H.ndim != len(shape) or tuple(int(n) for n in H.shape) != shape:
            raise ValueError(f"filter must have the shape {list(shape)}")
        if _dtype_name(H) != ("complex64" if self.real == "float32" else "complex128"):
            raise ValueError("filter dtype does not match the convolver")
        _check(library().neo_b200_conv_stage_filter(self._h, _ptr(H), _space(H)))

    def stage_impulse(self, ir) -> None:
        """stage_filter(uniform_partition(ir, B)) for ir [C][taps] / [O][I][taps], B <= taps, num_partitions(taps, B) <= P; a shorter
        response is zero-padded to the handle's P partitions."""
        if self.cfg is None:
            raise RuntimeError("no filter set")
        lead = (int(self.cfg.outputs),) if self.topology == DIAGONAL else (int(self.cfg.outputs), int(self.cfg.inputs))
        if ir.ndim != len(lead) + 1 or tuple(int(n) for n in ir.shape[:-1]) != lead or _dtype_name(ir) != self.real:
            raise ValueError("impulse response shape/dtype mismatch")
        taps, block = int(ir.shape[-1]), int(self.cfg.block)
        if taps < block or num_partitions(taps, block) > self.cfg.partitions:
            raise ValueError(f"impulse response of {taps} taps does not fit {self.cfg.partitions} partitions of {block}")
        _check(library().neo_b200_conv_stage_impulse(self._h, _ptr(ir), taps, _space(ir)))

    def crossfade(self, fade: int, delay: int = 0) -> int:
        """Switch to the staged filter with a linear fade of `fade` samples (0: hard switch) that starts `delay` samples after the
        last sample delivered so far, inside any later call. Returns `start`, the absolute index (samples since the last reset /
        filter / impulse) of the fade's first sample (neo_b200_conv_crossfade)."""
        if self.cfg is None:
            raise RuntimeError("no filter set")
        if int(fade) < 0 or int(delay) < 0:
            raise ValueError("fade and delay must be >= 0")
        start = _sz(0)
        _check(library().neo_b200_conv_crossfade(self._h, int(delay), int(fade), C.byref(start)))
        return int(start.value)

    def set_stream(self, stream) -> None:
        self._stream = _stream_ptr(stream)
        if self._h:
            _check(library().neo_b200_conv_set_stream(self._h, self._stream))

    def synchronize(self) -> None:
        _check(library().neo_b200_conv_synchronize(self._h))

    def reset(self) -> None:
        _check(library().neo_b200_conv_reset(self._h))

    def profile(self, enable: bool) -> None:
        _check(library().neo_b200_conv_profile_enable(self._h, int(enable)))

    def profile_read(self, frame_phases: bool = False):
        """(ms_r2c, ms_mac, ms_c2r, mac_launches) since the last read; synchronises the stream. With frame_phases the tuple is
        (ms_r2c, ms_mac, ms_c2r, ms_frame_forward, ms_frame_inverse, mac_launches)."""
        ms = (C.c_double * 5)()
        n = C.c_uint64(0)
        _check(library().neo_b200_conv_profile_read(self._h, ms, C.byref(n)))
        if frame_phases:
            return float(ms[0]), float(ms[1]), float(ms[2]), float(ms[3]), float(ms[4]), int(n.value)
        return float(ms[0]), float(ms[1]), float(ms[2]), int(n.value)

    def device_bytes(self) -> int:
        return int(library().neo_b200_conv_device_bytes(self._h))

    def __call__(self, x, out=None):
        """convolver(block) for every channel: x[inputs][T*B] processed as T blocks; in place when out is None
        (diagonal only, like the reference)."""
        block = int(self.cfg.block)
        if x.ndim != 2 or x.shape[0] != self.cfg.inputs or x.shape[1] % block != 0 or _dtype_name(x) != self.real:
            raise ValueError(f"expected {self.real}[{self.cfg.inputs}][T*{block}]")
        if out is None:
            out = x if self.topology == DIAGONAL else _empty_like_kind(x, (int(self.cfg.outputs), x.shape[1]), self.real)
        _check(library().neo_b200_conv_process(self._h, _ptr(x), _ptr(out), x.shape[1] // block, _space(x)))
        return out

    # split form used around the cross-device reduction of partition-sharded handles
    def forward(self, x) -> None:
        block = int(self.cfg.block)
        _check(library().neo_b200_conv_forward(self._h, _ptr(x), x.shape[1] // block, _space(x)))

    def forward_range(self, x, first: int, count: int, final: bool) -> None:
        """forward() for channels [first, first+count) only; x is the whole [inputs][T*B] device array."""
        block = int(self.cfg.block)
        _check(library().neo_b200_conv_forward_range(self._h, _ptr(x), x.shape[1] // block, first, count, int(final)))

    def spectra_ptr(self) -> tuple[int, int]:
        p, n = _vp(), _sz(0)
        _check(library().neo_b200_conv_spectra(self._h, C.byref(p), C.byref(n)))
        return int(p.value), int(n.value)

    def spectra_tensor(self, blocks: int):
        """torch view [outputs][blocks][2B] (float32 pairs) of the partial spectra produced by forward()."""
        import torch

        ptr, _ = self.spectra_ptr()  # a partition-sharded handle alternates between two buffers: ask after every forward
        views = getattr(self, "_spectra_view", None)
        if not isinstance(views, dict):
            views = self._spectra_view = {}
        if (ptr, blocks) in views:
            return views[(ptr, blocks)]
        n = int(self.cfg.outputs) * blocks * int(self.cfg.block) * 2
        dt = np.float32 if self.real == "float32" else np.float64

        class _Raw:
            __cuda_array_interface__ = {"shape": (n,), "typestr": np.dtype(dt).str, "data": (ptr, False), "version": 3}

        view = torch.as_tensor(_Raw(), device=f"cuda:{torch.cuda.current_device()}").view(int(self.cfg.outputs), blocks, -1)
        views[(ptr, blocks)] = view
        return view

    def inverse(self, spectra, out, first: int, count: int, blocks: int) -> None:
        sp = spectra if isinstance(spectra, int) else _ptr(spectra)
        _check(library().neo_b200_conv_inverse(self._h, sp, _ptr(out), first, count, blocks, _space(out)))

    def close(self) -> None:
        if self._h:
            library().neo_b200_conv_destroy(self._h)
            self._h = _vp()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class LowLatencyConvolver:
    """A bank of upols_convolver instances at ONE block of latency for long impulse responses (include/neo_b200.h:
    neo_b200_lowlat_*): the first partitions run per block, later stretches in frame mode on side streams (non-uniform
    partitioning). `filter(H)` / `impulse(ir, block)`, then call on any whole number of blocks, or `process_samples` on any
    number of samples (each output returned by the call that delivers its input). `stage_filter(H)` / `stage_impulse(ir)` then
    `crossfade(fade)` switch to a new response mid-stream with a linear crossfade, keeping every delay line.

    frame_blocks: the level frame sizes T_1 < ... < T_n (powers of two in [2, 512], n <= 4); None = the library default.
    """

    def __init__(self, dtype="float32", frame_blocks=None):
        self.real = _REAL_OF[str(np.dtype(dtype))]
        self.frame_blocks = tuple(int(t) for t in frame_blocks) if frame_blocks else ()
        self._h = _vp()
        self.cfg = None
        self._stream = None

    @staticmethod
    def _config(dtype_code: int, channels: int, block: int, partitions: int, frame_blocks) -> LowLatConfig:
        fb = tuple(frame_blocks or ())
        arr = (_sz * 4)(*(list(fb[:4]) + [0] * (4 - len(fb[:4]))))  # more than 4 levels: the library reports it
        return LowLatConfig(dtype_code, channels, block, partitions, len(fb), arr)

    @staticmethod
    def layout(partitions: int, block: int, frame_blocks=None, dtype="float32") -> dict:
        """The schedule the library builds, without a device: {"frame_blocks": (T_1, ...), "head": (0, e),
        "levels": [(begin, end), ...]} -- levels that would start at or past `partitions` are dropped."""
        cfg = LowLatencyConvolver._config(_DTYPE_CODE[_REAL_OF[str(np.dtype(dtype))]], 1, block, partitions, frame_blocks)
        n = _sz(0)
        fb = (_sz * 4)()
        ranges = (_sz * 10)()
        _check(library().neo_b200_lowlat_layout(C.byref(cfg), C.byref(n), fb, ranges))
        n = int(n.value)
        return {
            "frame_blocks": tuple(int(fb[i]) for i in range(n)),
            "head": (int(ranges[0]), int(ranges[1])),
            "levels": [(int(ranges[2 + 2 * i]), int(ranges[3 + 2 * i])) for i in range(n)],
        }

    def _create(self, channels, block, partitions):
        self.close()
        self.cfg = self._config(_DTYPE_CODE[self.real], channels, block, partitions, self.frame_blocks)
        _check(library().neo_b200_lowlat_create(C.byref(self._h), C.byref(self.cfg)))
        if self._stream is not None:
            _check(library().neo_b200_lowlat_set_stream(self._h, self._stream))

    def filter(self, H) -> None:
        """H [C][P][B+1] (uniform_partition layout): deep copy, state zeroed."""
        if H.ndim != 3:
            raise ValueError("filter must be [channels][partitions][block+1]")
        if _dtype_name(H) != ("complex64" if self.real == "float32" else "complex128"):
            raise ValueError("filter dtype does not match the convolver")
        self._create(int(H.shape[0]), int(H.shape[2]) - 1, int(H.shape[1]))
        _check(library().neo_b200_lowlat_set_filter(self._h, _ptr(H), _space(H)))

    def impulse(self, ir, block: int) -> None:
        """filter(uniform_partition(ir, block)) without materialising H on the host. ir: [C][L]."""
        if ir.ndim != 2 or _dtype_name(ir) != self.real:
            raise ValueError("impulse response shape/dtype mismatch")
        taps = int(ir.shape[1])
        self._create(int(ir.shape[0]), block, num_partitions(taps, block))
        _check(library().neo_b200_lowlat_set_impulse(self._h, _ptr(ir), taps, _space(ir)))

    def stage_filter(self, H) -> None:
        """H [C][P][B+1] of this handle's shape, prepared next to the current filter for `crossfade`: no output, delay line or
        position changes (neo_b200_lowlat_stage_filter)."""
        if self.cfg is None:
            raise RuntimeError("no filter set")
        shape = (int(self.cfg.channels), int(self.cfg.partitions), int(self.cfg.block) + 1)
        if H.ndim != 3 or tuple(int(n) for n in H.shape) != shape:
            raise ValueError(f"filter must be [{shape[0]}][{shape[1]}][{shape[2]}]")
        if _dtype_name(H) != ("complex64" if self.real == "float32" else "complex128"):
            raise ValueError("filter dtype does not match the convolver")
        _check(library().neo_b200_lowlat_stage_filter(self._h, _ptr(H), _space(H)))

    def stage_impulse(self, ir) -> None:
        """stage_filter(uniform_partition(ir, B)) for ir [C][taps], B <= taps, num_partitions(taps, B) <= P; a shorter response
        is zero-padded to the handle's P partitions."""
        if self.cfg is None:
            raise RuntimeError("no filter set")
        if ir.ndim != 2 or ir.shape[0] != self.cfg.channels or _dtype_name(ir) != self.real:
            raise ValueError("impulse response shape/dtype mismatch")
        taps, block = int(ir.shape[1]), int(self.cfg.block)
        if taps < block or num_partitions(taps, block) > self.cfg.partitions:
            raise ValueError(f"impulse response of {taps} taps does not fit {self.cfg.partitions} partitions of {block}")
        _check(library().neo_b200_lowlat_stage_impulse(self._h, _ptr(ir), taps, _space(ir)))

    def crossfade(self, fade: int) -> int:
        """Switch to the staged filter with a linear fade of `fade` samples (0: hard switch). Returns `start`, the absolute index
        (samples since the last reset / filter / impulse) of the fade's first sample (neo_b200_lowlat_crossfade)."""
        if self.cfg is None:
            raise RuntimeError("no filter set")
        if int(fade) < 0:
            raise ValueError("fade must be >= 0")
        start = _sz(0)
        _check(library().neo_b200_lowlat_crossfade(self._h, int(fade), C.byref(start)))
        return int(start.value)

    def set_stream(self, stream) -> None:
        self._stream = _stream_ptr(stream)
        if self._h:
            _check(library().neo_b200_lowlat_set_stream(self._h, self._stream))

    def synchronize(self) -> None:
        _check(library().neo_b200_lowlat_synchronize(self._h))

    def reset(self) -> None:
        _check(library().neo_b200_lowlat_reset(self._h))

    def device_bytes(self) -> int:
        return int(library().neo_b200_lowlat_device_bytes(self._h))

    def __call__(self, x, out=None):
        """convolver(block) for every channel: x [C][n*B] processed as n blocks; in place when out is None."""
        if self.cfg is None:
            raise RuntimeError("no filter set")
        block = int(self.cfg.block)
        if x.ndim != 2 or x.shape[0] != self.cfg.channels or x.shape[1] % block != 0 or _dtype_name(x) != self.real:
            raise ValueError(f"expected {self.real}[{self.cfg.channels}][n*{block}]")
        if out is None:
            out = x
        _check(library().neo_b200_lowlat_process(self._h, _ptr(x), _ptr(out), x.shape[1] // block, _space(x)))
        return out

    def process_samples(self, x, out=None):
        """x [C][n], any n >= 1, returned in the same call: the handle keeps its position inside the current block, so a host
        whose buffer size changes from call to call needs no FIFO in front (neo_b200_lowlat_process_samples). In place when out
        is None."""
        if self.cfg is None:
            raise RuntimeError("no filter set")
        if x.ndim != 2 or x.shape[0] != self.cfg.channels or x.shape[1] < 1 or _dtype_name(x) != self.real:
            raise ValueError(f"expected {self.real}[{self.cfg.channels}][n], n >= 1")
        if out is None:
            out = x
        _check(library().neo_b200_lowlat_process_samples(self._h, _ptr(x), _ptr(out), x.shape[1], _space(x)))
        return out

    def close(self) -> None:
        if self._h:
            library().neo_b200_lowlat_destroy(self._h)
            self._h = _vp()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def bank_unique_id() -> bytes:
    """The 128-byte id rank 0 creates and hands to every rank of a rank-per-process Bank (out of band: torch.distributed, MPI ...)."""
    buf = C.create_string_buffer(BANK_ID_BYTES)
    _check(library().neo_b200_bank_unique_id(buf))
    return bytes(buf.raw)


def _info_dict(info: BankRankInfo) -> dict:
    return {name: int(getattr(info, name)) for name, _ in BankRankInfo._fields_}


class Bank:
    """One convolver bank spread over the GPUs of one box (neo_b200_bank_*, include/neo_b200.h): `layout = (channel_groups,
    partition_shards)`, rank = group * partition_shards + shard.

    All ranks in this process:  Bank(..., layout=(Gc, Gp), devices=[0, 1, ...])   (peer-memory transport)
    One rank per process:       Bank(..., layout=(Gc, Gp), rank=r, world=N, unique_id=id, device=local)   (NCCL transport)

    `ranks` lists what each LOCAL rank holds and moves (BankRankInfo as dicts). Buffers: one array for the whole process
    ([rows of all local ranks][T*B], local ranks ascending) or a list with one array per local rank."""

    def __init__(self, kind: int, dtype, topology: int, outputs: int, inputs: int, block: int, partitions: int, max_blocks: int = 1,
                 frame_blocks: int = 0, layout=(1, 1), devices=None, rank=None, world=None, unique_id=None, device=None):
        self.real = _REAL_OF[str(np.dtype(dtype))]
        self.topology = topology
        inputs = outputs if topology == DIAGONAL else inputs
        self.cfg = ConvConfig(kind, _DTYPE_CODE[self.real], topology, outputs, inputs, block, partitions, frame_blocks or max_blocks, 0, 0,
                              frame_blocks, 0)
        self.layout = BankLayout(int(layout[0]), int(layout[1]))
        self._h = _vp()
        lib = library()
        if devices is not None:
            dev = (_i * len(devices))(*[int(d) for d in devices])
            _check(lib.neo_b200_bank_create(C.byref(self._h), C.byref(self.cfg), C.byref(self.layout), dev, len(devices)))
        else:
            uid = C.create_string_buffer(unique_id, BANK_ID_BYTES) if unique_id is not None else None
            _check(lib.neo_b200_bank_create_rank(C.byref(self._h), C.byref(self.cfg), C.byref(self.layout), int(device or 0), int(rank),
                                                 int(world), uid))
        n = _sz(0)
        _check(lib.neo_b200_bank_local_ranks(self._h, C.byref(n)))
        self.ranks = []
        for l in range(int(n.value)):
            info = BankRankInfo()
            _check(lib.neo_b200_bank_local_rank(self._h, l, C.byref(info)))
            self.ranks.append(_info_dict(info))

    @staticmethod
    def layout_info(kind, dtype, topology, outputs, inputs, block, partitions, max_blocks, frame_blocks, layout, rank: int) -> dict:
        real = _REAL_OF[str(np.dtype(dtype))]
        inputs = outputs if topology == DIAGONAL else inputs
        cfg = ConvConfig(kind, _DTYPE_CODE[real], topology, outputs, inputs, block, partitions, frame_blocks or max_blocks, 0, 0, frame_blocks, 0)
        lay = BankLayout(int(layout[0]), int(layout[1]))
        info = BankRankInfo()
        _check(library().neo_b200_bank_layout_info(C.byref(cfg), C.byref(lay), rank, C.byref(info)))
        return _info_dict(info)

    def _per_rank(self, arrays, key_first: str, key_count: str, what: str):
        """one pointer per local rank from a list of arrays, or from one array holding the rows of all local ranks in rank order"""
        if isinstance(arrays, (list, tuple)):
            if len(arrays) != len(self.ranks):
                raise ValueError(f"{what}: expected {len(self.ranks)} arrays, one per local rank")
            for a, r in zip(arrays, self.ranks):
                if a.shape[0] != r[key_count]:
                    raise ValueError(f"{what}: rank {r['rank']} moves {r[key_count]} rows, got {a.shape[0]}")
            return (_vp * len(arrays))(*[_ptr(a) for a in arrays]), _space(arrays[0]), arrays
        total = sum(r[key_count] for r in self.ranks)
        if arrays.shape[0] != total:
            raise ValueError(f"{what}: expected {total} rows (those of the local ranks), got {arrays.shape[0]}")
        if _is_device(arrays) and len(self.ranks) > 1:
            raise ValueError(f"{what}: device buffers of a multi-rank process must be given per rank (each on its own device)")
        base, row_bytes = _ptr(arrays), int(np.prod(arrays.shape[1:])) * (4 if self.real == "float32" else 8) * (2 if "complex" in _dtype_name(arrays) else 1)
        first0 = self.ranks[0][key_first]
        ptrs = [base + (r[key_first] - first0) * row_bytes for r in self.ranks]
        return (_vp * len(ptrs))(*ptrs), _space(arrays), arrays

    def impulse(self, ir) -> None:
        """ir: one array PER LOCAL RANK with the impulse responses of that rank's channel group ([group_count][taps], matrix topology
        [group_count][inputs][taps]); the partition shards of one group each get the group's rows. HOST arrays, or DEVICE arrays on the
        rank's own device."""
        arrs = ir if isinstance(ir, (list, tuple)) else [ir]
        if len(arrs) != len(self.ranks):
            raise ValueError(f"expected {len(self.ranks)} impulse-response arrays, one per local rank")
        taps = int(arrs[0].shape[-1])
        ptrs = (_vp * len(arrs))(*[_ptr(a) for a in arrs])
        _check(library().neo_b200_bank_set_impulse(self._h, ptrs, taps, _space(arrs[0])))

    def impulse_global(self, ir) -> None:
        """ir: the impulse responses of the WHOLE bank on the host ([channels][taps] / [outputs][inputs][taps]); every local rank takes
        its group's rows."""
        self.impulse([np.ascontiguousarray(ir[r["group_first"] : r["group_first"] + r["group_count"]]) for r in self.ranks])

    def filter_global(self, H) -> None:
        arrs = [np.ascontiguousarray(H[r["group_first"] : r["group_first"] + r["group_count"]]) for r in self.ranks]
        ptrs = (_vp * len(arrs))(*[_ptr(a) for a in arrs])
        _check(library().neo_b200_bank_set_filter(self._h, ptrs, HOST))

    def reset(self) -> None:
        _check(library().neo_b200_bank_reset(self._h))

    def submit(self, x, out) -> None:
        first = x[0] if isinstance(x, (list, tuple)) else x
        blocks = int(first.shape[1]) // int(self.cfg.block)
        xin, space, keep_x = self._per_rank(x, "in_first", "in_count", "input")
        yout, space_o, keep_y = self._per_rank(out, "out_first", "out_count", "output")
        if space != space_o:
            raise ValueError("input and output must live in the same memory space")
        self._keep = (keep_x, keep_y, getattr(self, "_keep", None) and self._keep[:2])  # buffers of the steps in flight stay alive
        _check(library().neo_b200_bank_submit(self._h, xin, yout, blocks, space))

    def wait(self) -> None:
        _check(library().neo_b200_bank_wait(self._h))

    def __call__(self, x, out):
        first = x[0] if isinstance(x, (list, tuple)) else x
        blocks = int(first.shape[1]) // int(self.cfg.block)
        xin, space, _ = self._per_rank(x, "in_first", "in_count", "input")
        yout, _, _ = self._per_rank(out, "out_first", "out_count", "output")
        _check(library().neo_b200_bank_process(self._h, xin, yout, blocks, space))
        return out

    def timer_start(self) -> None:
        _check(library().neo_b200_bank_timer_start(self._h))

    def timer_stop(self) -> float:
        """milliseconds of device time since timer_start (CUDA events on the bank's streams, longest local rank); waits for all steps"""
        ms = C.c_double(0.0)
        _check(library().neo_b200_bank_timer_stop(self._h, C.byref(ms)))
        return float(ms.value)

    def profile(self, enable: bool) -> None:
        _check(library().neo_b200_bank_profile_enable(self._h, int(enable)))

    def profile_read(self, local_index: int = 0):
        """(ms_r2c, ms_mac, ms_c2r, ms_frame_forward, ms_frame_inverse, mac_launches) of one local rank since the last read"""
        ms = (C.c_double * 5)()
        n = C.c_uint64(0)
        _check(library().neo_b200_bank_profile_read(self._h, local_index, ms, C.byref(n)))
        return float(ms[0]), float(ms[1]), float(ms[2]), float(ms[3]), float(ms[4]), int(n.value)

    def device_bytes(self, local_index: int = 0) -> int:
        return int(library().neo_b200_bank_device_bytes(self._h, local_index))

    def close(self) -> None:
        if self._h:
            library().neo_b200_bank_destroy(self._h)
            self._h = _vp()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


# ---- free functions with the reference's Python names (extra/python/src/neo/fft/__init__.py:20-29) -----------------------
def _norm_factor(norm: str, n: int, forward: bool) -> float:
    # extra/python/src/main.cpp:150-162
    if norm == "backward":
        return 1.0 if forward else 1.0 / n
    if norm == "ortho":
        return 1.0 / np.sqrt(n)
    if norm == "forward":
        return 1.0 / n if forward else 1.0
    raise RuntimeError(f"unsupported norm '{norm}'")


def _c2c(x, n, norm, direction):
    x = np.asarray(x)
    if x.dtype not in (np.complex64, np.complex128):
        x = x.astype(np.complex128 if x.dtype == np.float64 else np.complex64)
    n = x.shape[-1] if n is None else n
    if n & (n - 1) != 0 or n == 0:
        raise RuntimeError("only power-of-two sizes are supported")  # main.cpp:137-139
    if x.shape[-1] != n:
        buf = np.zeros(x.shape[:-1] + (n,), dtype=x.dtype)
        m = min(n, x.shape[-1])
        buf[..., :m] = x[..., :m]
        x = buf
    else:
        x = np.ascontiguousarray(x).copy()
    plan = FFTPlan(n.bit_length() - 1, x.dtype)
    plan(x, direction)
    plan.close()
    scale = _norm_factor(norm, n, direction == FORWARD)
    return x if scale == 1.0 else (x * x.real.dtype.type(scale)).astype(x.dtype)


def rfftfreq(size: int, inv_sample_rate: float, dtype="float32") -> np.ndarray:
    """neo::rfftfreq (fft/rfftfreq.hpp:12-29): out[i] = i * (1 / inv_sample_rate) * (1 / size) for i < size, evaluated in `dtype`
    in the reference's order (host-side index helper, no transform involved)."""
    real = np.dtype(dtype).type
    fs = real(1) / real(inv_sample_rate)
    inv_size = real(1) / real(size)
    return (np.arange(size).astype(real) * fs * inv_size).astype(real)


def fft(x, n=None, norm="backward"):
    return _c2c(x, n, norm, FORWARD)


def ifft(x, n=None, norm="backward"):
    return _c2c(x, n, norm, BACKWARD)


def rfft(x):
    x = np.ascontiguousarray(x)
    plan = RFFTPlan(int(x.shape[-1]).bit_length() - 1, x.dtype)
    out = plan.rfft(x)
    plan.close()
    return out


def irfft(x, n: int):
    x = np.ascontiguousarray(x)
    plan = RFFTPlan(int(n).bit_length() - 1, _REAL_OF[str(x.dtype)])
    out = plan.irfft(x)
    plan.close()
    return out


def fft_convolve(signal, patch):
    """neo::convolution::fft_convolve (convolution/fft_convolver.hpp:84-93), mode::full, batched over leading axes:
    signal[..., n] * patch[..., m] -> [..., n + m - 1]."""
    real = _dtype_name(signal)
    if _dtype_name(patch) != real or signal.shape[:-1] != patch.shape[:-1]:
        raise ValueError("signal and patch must share dtype and batch shape")
    n, m = int(signal.shape[-1]), int(patch.shape[-1])
    batch = int(np.prod(signal.shape[:-1], dtype=np.int64)) if signal.ndim > 1 else 1
    if n == 0 or m == 0:
        return _empty_like_kind(signal, tuple(signal.shape[:-1]) + (0,), real)  # fft_convolver.hpp:88-90
    h = _vp()
    _check(library().neo_b200_fft_convolver_create(C.byref(h), n, m, _DTYPE_CODE[real]))
    try:
        out = _empty_like_kind(signal, tuple(signal.shape[:-1]) + (n + m - 1,), real)
        if _space(signal) == DEVICE:
            import torch

            torch.cuda.synchronize()  # the handle runs on its own stream: the inputs must be complete
        _check(library().neo_b200_fft_convolver_exec(h, _ptr(signal), _ptr(patch), _ptr(out), batch, _space(signal)))
        if _space(signal) == DEVICE:
            import torch

            torch.cuda.synchronize()  # the handle (and its stream) is destroyed below
    finally:
        library().neo_b200_fft_convolver_destroy(h)
    return out


def convolve(in1, in2, mode: str = "full", method: str = "upols", block: int | None = None):
    """neo.convolve (extra/python/src/main.cpp:171-198): full linear convolution of two 1-D signals. The reference binds
    method="direct"/"fft"; the partitioned methods of convolution/method.hpp:8-17 ("upols", "upola") are what runs here."""
    if mode != "full":
        raise RuntimeError(f"unsupported mode '{mode}'")  # main.cpp:197, asserted by extra/python/test/test.py:36-40
    if method not in ("upols", "upola", "ols", "ola", "fft", "auto"):
        raise RuntimeError(f"unsupported method '{method}'")
    sig = np.ascontiguousarray(in1, dtype=np.float32)
    ir = np.ascontiguousarray(in2, dtype=np.float32)
    if sig.ndim != 1 or ir.ndim != 1:
        raise RuntimeError("unsupported ndim")  # main.cpp:126
    if sig.size == 0 or ir.size == 0:
        return np.zeros(0, dtype=np.float32)
    if method == "fft":  # main.cpp:190-192: fft_convolve
        return fft_convolve(sig, ir)
    if block is None:
        block = max(2, min(4096, 1 << max(1, (ir.size - 1).bit_length())))
    total = sig.size + ir.size - 1
    taps = max(ir.size, block)
    ir_p = np.zeros((1, taps), dtype=np.float32)
    ir_p[0, : ir.size] = ir
    blocks = -(-total // block)
    x = np.zeros((1, blocks * block), dtype=np.float32)
    x[0, : sig.size] = sig
    conv = Convolver(UPOLA if method in ("upola", "ola") else UPOLS, "float32", DIAGONAL, max_blocks=min(blocks, 64))
    conv.impulse(ir_p, block)
    step = conv.max_blocks * block
    for s in range(0, x.shape[1], step):
        chunk = np.ascontiguousarray(x[:, s : s + step])
        conv(chunk)
        x[:, s : s + step] = chunk
    conv.close()
    return x[0, :total].copy()
