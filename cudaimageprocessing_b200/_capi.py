"""ctypes view of the C ABI in include/gf_b200.h.  Pointers are plain integers (device
addresses from torch's `data_ptr()`); nothing here touches image data."""
from __future__ import annotations

import ctypes
from ctypes import c_float, c_int, c_int64, c_size_t, c_void_p

GF_OK, GF_ERR_INVALID, GF_ERR_UNSUPPORTED, GF_ERR_CUDA, GF_ERR_NOMEM = range(5)
BORDER_REFLECT101, BORDER_TRUNCATE, BORDER_REFLECT = 0, 1, 2

# every symbol include/gf_b200.h declares: name -> (restype, argtypes)
P = c_void_p
SIGNATURES = {
    "gf_last_error": (ctypes.c_char_p, []),
    "gf_version": (c_int, []),
    "gf_device_info": (c_int, [P, P, P]),
    "gf_create": (c_int, [P, c_int, c_int, c_int, c_int]),
    "gf_run": (c_int, [P, P, P, P, c_int, c_float, c_int, c_int64, c_int64, c_int64, P]),
    "gf_destroy": (c_int, [P]),
    "gf_guided_gray": (c_int, [P, P, P, P, P, c_int, c_int, c_int64, c_int64, c_int64, c_int64, c_int, c_float, c_int, P]),
    "gf_guided_color": (c_int, [P, P, P, c_int, c_int, c_int, c_int64, c_int64, c_int64, c_int, c_float, c_int, P]),
    "gf_fast_guided_gray": (c_int, [P, P, P, c_int, c_int, c_int64, c_int64, c_int64, c_int, c_float, c_int, c_int, P]),
    "gf_fast_guided_gray_u8": (c_int, [P, P, P, c_int, c_int, c_int64, c_int64, c_int64, c_int, c_float, c_int, c_int, P]),
    "gf_fast_guided_color": (c_int, [P, P, P, c_int, c_int, c_int, c_int64, c_int64, c_int64, c_int, c_float, c_int, c_int,
                                     P]),
    "gf_guided_batch": (c_int, [P, P, P, c_int, c_int, c_int, c_int, c_int64, c_int64, c_int64, c_int64, c_int64, c_int64,
                                c_int, c_float, c_int, P]),
    "gf_guided_gray_strip": (c_int, [P, P, P, c_int, c_int, c_int, c_int, c_int, c_int, c_int64, c_int64, c_int64,
                                     c_int, c_float, c_int, P]),
    "gf_strip_layout": (c_int, [c_int, c_int, c_int, c_int, P, P]),
    "gf_run_strips": (c_int, [P, P, P, c_int, c_int, c_int, c_int, c_int64, c_int64, c_int64, c_int, c_float, c_int, P, P, P]),
    "gf_device_alloc": (c_int, [P, c_size_t]),
    "gf_device_free": (c_int, [P]),
    "gf_ipc_export": (c_int, [P, P]),
    "gf_ipc_open": (c_int, [P, P]),
    "gf_ipc_close": (c_int, [P]),
    "gf_window_sums_u8": (c_int, [P, P, P, P, P, P, c_int, c_int, c_int64, c_int64, c_int, c_int, P]),
    "gf_box_filter": (c_int, [P, P, c_int, c_int, c_int, c_int64, c_int64, c_int, c_int, P]),
    "gf_multiply": (c_int, [P, P, P, c_int, c_int, c_int, c_int, c_int64, c_int64, P]),
    "gf_calc_a": (c_int, [P, P, P, P, P, c_int, c_int, c_int, c_int, c_int64, c_int64, c_float, P]),
    "gf_calc_b": (c_int, [P, P, P, P, c_int, c_int, c_int, c_int, c_int64, c_int64, P]),
    "gf_linear_transform": (c_int, [P, P, P, P, c_int, c_int, c_int, c_int, c_int64, c_int64, P]),
    "gf_guided_gray_host": (c_int, [P, P, P, c_int, c_int, c_int, c_float, c_int]),
    "gf_host_alloc": (c_int, [P, c_size_t]),
    "gf_host_register": (c_int, [P, c_size_t]),
    "gf_host_unregister": (c_int, [P]),
    "gf_host_free": (c_int, [P]),
    "gf_guided_gray_u8": (c_int, [P, P, P, c_int, c_int, c_int64, c_int64, c_int64, c_int, c_float, c_int, P]),
    "gf_guided_color_u8": (c_int, [P, P, P, c_int, c_int, c_int, c_int64, c_int64, c_int64, c_int, c_float, c_int, P]),
    "gf_guided_per_channel_u8": (c_int, [P, P, P, c_int, c_int, c_int, c_int64, c_int64, c_int64, c_int, c_float, c_int, P]),
    "gf_gaussian_gray": (c_int, [P, P, c_int, c_int, c_int64, c_int64, c_int, ctypes.c_double, P]),
    "gf_integral_u8_i32": (c_int, [P, P, P, c_int, c_int, c_int64, c_int64, P]),
    "gf_integral_u8_i64": (c_int, [P, P, P, c_int, c_int, c_int64, c_int64, P]),
    "gf_integral_u8_i32_padded": (c_int, [P, P, c_int, c_int, c_int64, c_int, c_int, P]),
    "gf_last_kernel": (ctypes.c_char_p, []),
    "gf_launch_count": (c_int64, []),
    "gf_set_option": (c_int, [ctypes.c_char_p, c_int]),
}


class StripPeer(ctypes.Structure):
    """gf_strip_peer (include/gf_b200.h): a neighbour's strip buffers as seen from this device."""
    _fields_ = [("guide", P), ("src", P), ("guide_stride", c_int64), ("src_stride", c_int64), ("top", c_int), ("rows", c_int)]


class GfError(RuntimeError):
    def __init__(self, status: int, message: str):
        super().__init__(f"gf status {status}: {message}")
        self.status = status


class GfApi:
    """Typed wrapper over a loaded library exporting the gf_* C ABI."""

    def __init__(self, cdll: ctypes.CDLL):
        self.cdll = cdll
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(cdll, name)          # AttributeError if the library lacks a declared symbol
            fn.restype = res
            fn.argtypes = args

    def _check(self, status: int):
        if status != GF_OK:
            raise GfError(status, self.cdll.gf_last_error().decode())

    def call(self, name: str, *args):
        self._check(getattr(self.cdll, name)(*args))

    def set_option(self, name: str, value: int):
        """Developer/test knob of the launch paths (include/gf_b200.h: gf_set_option); value < 0 = default."""
        self.call("gf_set_option", name.encode(), int(value))

    def last_kernel(self) -> str:
        return self.cdll.gf_last_kernel().decode()

    def launch_count(self) -> int:
        return int(self.cdll.gf_launch_count())

    def device_info(self):
        a, b, c = c_int(), c_int(), c_int()
        self.call("gf_device_info", ctypes.addressof(a), ctypes.addressof(b), ctypes.addressof(c))
        return a.value, b.value, c.value
