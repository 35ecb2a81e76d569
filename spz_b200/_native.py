"""ctypes view of the C-ABI (include/spz_b200.h).  Loads spz_b200/_lib/libspz_b200.so.

There is no fallback: if the library is missing (and cannot be built because nvcc is absent) the
import of anything that needs it raises, and every codec call needs a CUDA device.
"""
from __future__ import annotations

import ctypes as C
import os

from . import build as _build

_f32p = C.POINTER(C.c_float)
_u8p = C.POINTER(C.c_uint8)


class Cloud(C.Structure):
    """SpzB200Cloud: float planes (GaussianCloud, splat-types.h:90-115)."""
    _fields_ = [("num_points", C.c_int64), ("sh_degree", C.c_int32), ("reserved", C.c_int32),
                ("positions", C.c_void_p), ("scales", C.c_void_p), ("rotations", C.c_void_p),
                ("alphas", C.c_void_p), ("colors", C.c_void_p), ("sh", C.c_void_p)]


class Packed(C.Structure):
    """SpzB200Packed: byte planes (PackedGaussians, load-spz.h:42-59)."""
    _fields_ = [("num_points", C.c_int64), ("sh_degree", C.c_int32),
                ("fractional_bits", C.c_int32), ("version", C.c_int32), ("reserved", C.c_int32),
                ("positions", C.c_void_p), ("scales", C.c_void_p), ("rotations", C.c_void_p),
                ("alphas", C.c_void_p), ("colors", C.c_void_p), ("sh", C.c_void_p)]


class PlyRows(C.Structure):
    """SpzB200PlyRows: row-major .ply vertex records + the column map."""
    _fields_ = [("num_points", C.c_int64), ("width", C.c_int32), ("sh_degree", C.c_int32), ("rows", C.c_void_p),
                ("col_pos", C.c_int32 * 3), ("col_scale", C.c_int32 * 3), ("col_rot", C.c_int32 * 4), ("col_alpha", C.c_int32),
                ("col_color", C.c_int32 * 3), ("col_rest", C.c_int32 * 45)]


class Timings(C.Structure):
    _fields_ = [("h2d_ms", C.c_double), ("kernel_ms", C.c_double), ("d2h_ms", C.c_double),
                ("wall_ms", C.c_double), ("h2d_bytes", C.c_int64), ("d2h_bytes", C.c_int64),
                ("kernel_launches", C.c_int32), ("chunks", C.c_int32), ("host_copy_ms", C.c_double),
                ("staged", C.c_int32), ("reserved", C.c_int32)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


OK, ERR_INVALID, ERR_NO_DEVICE, ERR_CUDA, ERR_NOMEM = 0, -1, -2, -3, -4

# every symbol include/spz_b200.h declares: name -> (restype, argtypes)
SIGNATURES = {
    "spzb200_create": (C.c_int, [C.c_int32, C.POINTER(C.c_void_p)]),
    "spzb200_destroy": (None, [C.c_void_p]),
    "spzb200_acquire": (C.c_int, [C.c_int32, C.POINTER(C.c_void_p)]),
    "spzb200_release": (None, [C.c_void_p]),
    "spzb200_unpack_records_host": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_int32, _f32p, C.c_void_p]),
    "spzb200_unpack_gather_host": (C.c_int, [C.c_void_p, C.POINTER(Packed), C.c_void_p, C.c_int64, _f32p, C.c_void_p]),
    "spzb200_unpack_gather_device": (C.c_int, [C.c_void_p, C.POINTER(Packed), C.c_void_p, C.c_int64, _f32p, C.c_void_p, C.c_void_p]),
    "spzb200_encode_device": (C.c_int, [C.c_void_p, C.POINTER(Cloud), C.c_int32, C.POINTER(Packed), C.c_void_p]),
    "spzb200_encode_device_as": (C.c_int, [C.c_void_p, C.POINTER(Cloud), C.c_int32, C.c_int32, C.POINTER(Packed), C.c_void_p]),
    "spzb200_encode_host_as": (C.c_int, [C.c_void_p, C.POINTER(Cloud), C.c_int32, C.c_int32, C.POINTER(Packed), C.POINTER(Timings)]),
    "spzb200_decode_device": (C.c_int, [C.c_void_p, C.POINTER(Packed), C.c_int32, C.POINTER(Cloud), C.c_void_p]),
    "spzb200_quantize_device": (C.c_int, [C.c_void_p, C.POINTER(Cloud), C.c_int32, C.c_int32, C.c_int32, C.POINTER(Cloud), C.c_void_p]),
    "spzb200_encode_host": (C.c_int, [C.c_void_p, C.POINTER(Cloud), C.c_int32, C.POINTER(Packed), C.POINTER(Timings)]),
    "spzb200_decode_host": (C.c_int, [C.c_void_p, C.POINTER(Packed), C.c_int32, C.POINTER(Cloud), C.POINTER(Timings)]),
    "spzb200_encode_ply_device": (C.c_int, [C.c_void_p, C.POINTER(PlyRows), C.c_int32, C.POINTER(Packed), C.c_void_p]),
    "spzb200_encode_ply_host": (C.c_int, [C.c_void_p, C.POINTER(PlyRows), C.c_int32, C.POINTER(Packed), C.POINTER(Timings)]),
    "spzb200_decode_ply_device": (C.c_int, [C.c_void_p, C.POINTER(Packed), C.c_int32, C.POINTER(PlyRows), C.c_void_p]),
    "spzb200_decode_ply_host": (C.c_int, [C.c_void_p, C.POINTER(Packed), C.c_int32, C.POINTER(PlyRows), C.POINTER(Timings)]),
    "spzb200_encode_host_multi": (C.c_int, [C.POINTER(C.c_int32), C.c_int32, C.POINTER(Cloud), C.c_int32, C.POINTER(Packed), C.POINTER(Timings)]),
    "spzb200_decode_host_multi": (C.c_int, [C.POINTER(C.c_int32), C.c_int32, C.POINTER(Packed), C.c_int32, C.POINTER(Cloud), C.POINTER(Timings)]),
    "spzb200_alloc_pinned": (C.c_int, [C.c_size_t, C.POINTER(C.c_void_p)]),
    "spzb200_free_pinned": (None, [C.c_void_p]),
    "spzb200_gzip": (C.c_int, [C.c_void_p, C.c_size_t, C.c_int32, C.POINTER(C.c_void_p), C.POINTER(C.c_size_t)]),
    "spzb200_gunzip": (C.c_int, [C.c_void_p, C.c_size_t, C.c_int32, C.POINTER(C.c_void_p), C.POINTER(C.c_size_t)]),
    "spzb200_free": (None, [C.c_void_p]),
    "spzb200_gzip_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.POINTER(C.c_void_p), C.POINTER(C.c_size_t), C.c_void_p]),
    "spzb200_save_spz_device": (C.c_int, [C.c_void_p, C.POINTER(Cloud), C.c_int32, C.c_int32, C.POINTER(C.c_void_p), C.POINTER(C.c_size_t),
                                          C.c_void_p]),
    "spzb200_spz_info": (C.c_int, [C.c_void_p, C.c_size_t, C.POINTER(C.c_int64), C.POINTER(C.c_int32)]),
    "spzb200_load_spz_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_int32, C.POINTER(Cloud), C.POINTER(C.c_int32), C.c_void_p]),
    "spzb200_gzip_table_info": (C.c_int, [C.c_void_p, C.c_size_t, C.POINTER(C.c_uint64), C.POINTER(C.c_int64)]),
    "spzb200_gunzip_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.POINTER(C.c_size_t),
                                        C.POINTER(C.c_int32), C.c_void_p]),
    "spzb200_gzip_device_batch": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]),
    "spzb200_save_spz_device_batch": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "spzb200_gunzip_device_batch": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                              C.c_void_p, C.c_void_p]),
    "spzb200_load_spz_device_batch": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p,
                                                C.c_void_p]),
    "spzb200_shard_range": (C.c_int, [C.c_int64, C.c_int32, C.c_int32, C.c_int32, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "spzb200_tile_gaussians": (C.c_int32, [C.c_int32]),
    "spzb200_flip_bits": (None, [C.c_int32, C.c_int32, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]),
    "spzb200_get_tables": (C.c_int, [C.c_void_p, _f32p, _f32p]),
    "spzb200_build_tables": (C.c_int, [_f32p, _f32p]),
    "spzb200_selfcheck_division": (C.c_int, [C.c_void_p, C.c_int32, C.c_uint64, C.c_uint64, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]),
    "spzb200_info": (C.c_int, [C.c_void_p, C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.POINTER(C.c_int64)]),
    "spzb200_set_force_generic": (None, [C.c_void_p, C.c_int32]),
    "spzb200_set_pack_mode": (None, [C.c_void_p, C.c_int32]),
    "spzb200_set_chunk_points": (None, [C.c_void_p, C.c_int64]),
    "spzb200_set_host_staging": (None, [C.c_void_p, C.c_int32, C.c_int32]),
    "spzb200_last_error": (C.c_char_p, []),
    "spzb200_version": (C.c_int32, []),
}

_lib = None


class NativeLibraryError(RuntimeError):
    pass


def lib() -> C.CDLL:
    """The loaded library; builds it first if it is missing or stale and nvcc is available."""
    global _lib
    if _lib is not None:
        return _lib
    path = _build.LIB
    variant = os.environ.get("SPZB200_LIB")  # a tuning variant built by scripts/ (development only)
    if variant:
        if not os.path.exists(variant):
            raise NativeLibraryError(f"SPZB200_LIB={variant} does not exist")
        path = variant
    elif not os.path.exists(path) or (not _build.up_to_date() and os.environ.get("SPZB200_NO_REBUILD") is None):
        try:
            _build.build()
        except Exception as e:  # noqa: BLE001
            if not os.path.exists(path):
                raise NativeLibraryError(
                    f"spz_b200: native library {path} is missing and could not be built ({e}); "
                    "there is no Python/CPU fallback for the codec") from e
    L = C.CDLL(path)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(L, name)  # AttributeError here = header and library disagree
        fn.restype, fn.argtypes = res, args
    _lib = L
    return L


def last_error() -> str:
    return lib().spzb200_last_error().decode("utf-8", "replace")


class CodecError(RuntimeError):
    def __init__(self, code: int, message: str, failed=()):
        super().__init__(f"spz_b200 error {code}: {message}")
        self.code = code
        self.failed = list(failed)  # batch calls: the indices of the inputs that failed


def check(rc: int) -> None:
    if rc != OK:
        raise CodecError(rc, last_error())
