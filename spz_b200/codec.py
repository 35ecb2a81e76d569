"""Plane-level front end of the C-ABI for torch tensors (device or pinned host) and numpy arrays.

PyTorch is used only for memory and streams; every byte of codec work happens inside
libspz_b200.so's sm_100a kernels.  This module mirrors the two hot-path functions of the
reference one to one:

    Context.encode_*  <->  spz::packGaussians    (load-spz.cc:257-331)
    Context.decode_*  <->  spz::unpackGaussians  (load-spz.cc:467-531)
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field
from typing import Any, Optional

import numpy as np

from . import _native as N

SH_DIM = {0: 0, 1: 3, 2: 8, 3: 15}

# floats (resp. bytes) per gaussian of each plane, in struct order
def float_plane_widths(sh_degree: int):
    return (3, 3, 4, 1, 3, 3 * SH_DIM[sh_degree])


def byte_plane_widths(sh_degree: int, version: int = 3):
    return (6 if version in (1, 4) else 9, 3, 4 if version >= 3 else 3, 1, 3, 3 * SH_DIM[sh_degree])


def float_bytes_per_gaussian(sh_degree: int) -> int:
    return 4 * sum(float_plane_widths(sh_degree))


def packed_bytes_per_gaussian(sh_degree: int, version: int = 3) -> int:
    return sum(byte_plane_widths(sh_degree, version))


def algorithmic_bytes_per_gaussian(sh_degree: int, version: int = 3) -> int:
    """Bytes a codec pass must move per gaussian: 301 at SH degree 3 (SURVEY.md section 8d)."""
    return float_bytes_per_gaussian(sh_degree) + packed_bytes_per_gaussian(sh_degree, version)


PLANES = ("positions", "scales", "rotations", "alphas", "colors", "sh")


@dataclass
class CloudPlanes:
    """GaussianCloud (splat-types.h:90-115) as six flat float32 planes."""
    n: int
    sh_degree: int
    positions: Any
    scales: Any
    rotations: Any
    alphas: Any
    colors: Any
    sh: Any
    antialiased: bool = False

    def planes(self):
        return tuple(getattr(self, p) for p in PLANES)


@dataclass
class PackedPlanes:
    """PackedGaussians (load-spz.h:42-59) as six flat uint8 planes."""
    n: int
    sh_degree: int
    positions: Any
    scales: Any
    rotations: Any
    alphas: Any
    colors: Any
    sh: Any
    fractional_bits: int = 12
    version: int = 3
    antialiased: bool = False

    def planes(self):
        return tuple(getattr(self, p) for p in PLANES)


def _is_torch(x) -> bool:
    return type(x).__module__.startswith("torch")


def _ptr(x, want_dtype: str, count: int, on_device: Optional[bool], name: str) -> int:
    """Address of a contiguous plane, with the reference's size check (load-spz.cc:106-127)."""
    if x is None:
        if count == 0:
            return 0
        raise ValueError(f"{name}: plane is None but {count} elements are required")
    if _is_torch(x):
        import torch
        dt = torch.float32 if want_dtype == "f4" else torch.uint8
        if x.dtype != dt:
            raise TypeError(f"{name}: expected {dt}, got {x.dtype}")
        if not x.is_contiguous():
            raise ValueError(f"{name}: tensor must be contiguous")
        if x.numel() != count:
            raise ValueError(f"{name}: expected {count} elements, got {x.numel()}")
        if on_device is not None and x.is_cuda != on_device:
            raise ValueError(f"{name}: expected a {'CUDA' if on_device else 'host'} tensor")
        return x.data_ptr() if count else 0
    a = x
    dt = np.float32 if want_dtype == "f4" else np.uint8
    if not isinstance(a, np.ndarray) or a.dtype != dt:
        raise TypeError(f"{name}: expected a numpy {np.dtype(dt).name} array")
    if not a.flags.c_contiguous:
        raise ValueError(f"{name}: array must be C-contiguous")
    if a.size != count:
        raise ValueError(f"{name}: expected {count} elements, got {a.size}")
    if on_device:
        raise ValueError(f"{name}: numpy arrays live on the host; a CUDA tensor is required")
    return a.ctypes.data if count else 0


def _cloud_struct(c: CloudPlanes, on_device: Optional[bool]) -> N.Cloud:
    if c.sh_degree not in SH_DIM:
        raise ValueError(f"sh_degree {c.sh_degree} not in 0..3")
    s = N.Cloud()
    s.num_points, s.sh_degree = c.n, c.sh_degree
    for name, w in zip(PLANES, float_plane_widths(c.sh_degree)):
        setattr(s, name, _ptr(getattr(c, name), "f4", c.n * w, on_device, name))
    return s


def _packed_struct(p: PackedPlanes, on_device: Optional[bool]) -> N.Packed:
    if p.sh_degree not in SH_DIM:
        raise ValueError(f"sh_degree {p.sh_degree} not in 0..3")
    s = N.Packed()
    s.num_points, s.sh_degree = p.n, p.sh_degree
    s.fractional_bits, s.version = p.fractional_bits, p.version
    for name, w in zip(PLANES, byte_plane_widths(p.sh_degree, p.version)):
        setattr(s, name, _ptr(getattr(p, name), "u1", p.n * w, on_device, name))
    return s


def pinned_array(count: int, dtype) -> np.ndarray:
    """A page-locked numpy array (spzb200_alloc_pinned); freed when the array is collected."""
    import weakref
    dt = np.dtype(dtype)
    nbytes = int(count) * dt.itemsize
    if nbytes == 0:
        return np.empty(0, dt)
    ptr = C.c_void_p(None)
    N.check(N.lib().spzb200_alloc_pinned(nbytes, C.byref(ptr)))
    buf = (C.c_uint8 * nbytes).from_address(ptr.value)
    arr = np.frombuffer(buf, dtype=dt, count=int(count))
    weakref.finalize(buf, N.lib().spzb200_free_pinned, C.c_void_p(ptr.value))
    return arr


def alloc_cloud(n: int, sh_degree: int, device=None, pinned: bool = False, numpy_arrays: bool = False) -> CloudPlanes:
    ws = float_plane_widths(sh_degree)
    if numpy_arrays:
        mk = pinned_array if pinned else np.empty
        return CloudPlanes(n, sh_degree, *[mk(n * w, np.float32) for w in ws])
    import torch
    kw = dict(dtype=torch.float32, device=device) if device is not None else dict(dtype=torch.float32, pin_memory=pinned)
    return CloudPlanes(n, sh_degree, *[torch.empty(n * w, **kw) for w in ws])


def alloc_packed(n: int, sh_degree: int, version: int = 3, device=None, pinned: bool = False,
                 numpy_arrays: bool = False, fractional_bits: int = 12) -> PackedPlanes:
    ws = byte_plane_widths(sh_degree, version)
    if numpy_arrays:
        mk = pinned_array if pinned else np.empty
        planes = [mk(n * w, np.uint8) for w in ws]
    else:
        import torch
        kw = dict(dtype=torch.uint8, device=device) if device is not None else dict(dtype=torch.uint8, pin_memory=pinned)
        planes = [torch.empty(n * w, **kw) for w in ws]
    return PackedPlanes(n, sh_degree, *planes, fractional_bits=fractional_bits, version=version)


def _host_bytes_call(fn, data, threads: int) -> bytes:
    buf = np.frombuffer(data, np.uint8) if not isinstance(data, np.ndarray) else np.ascontiguousarray(data, np.uint8)
    out, size = C.c_void_p(None), C.c_size_t(0)
    N.check(fn(buf.ctypes.data if buf.size else None, buf.size, int(threads), C.byref(out), C.byref(size)))
    try:
        return C.string_at(out.value, size.value)
    finally:
        N.lib().spzb200_free(out)


def gzip_bytes(data, threads: int = 1) -> bytes:
    """The container's gzip stage on the host (spzb200_gzip): threads <= 1 is the reference's stream."""
    return _host_bytes_call(N.lib().spzb200_gzip, data, threads)


def gunzip_bytes(data, threads: int = 1) -> bytes:
    return _host_bytes_call(N.lib().spzb200_gunzip, data, threads)


def spz_info(blob):
    """(num_points, sh_degree) from the header of .spz bytes (spzb200_spz_info; inflates 16 bytes, no GPU)."""
    buf = np.frombuffer(blob, np.uint8) if not isinstance(blob, np.ndarray) else np.ascontiguousarray(blob, np.uint8)
    n, deg = C.c_int64(0), C.c_int32(0)
    N.check(N.lib().spzb200_spz_info(C.c_void_p(buf.ctypes.data if buf.size else None), buf.size, C.byref(n), C.byref(deg)))
    return n.value, deg.value


def gzip_table_info(blob):
    """(inflated_size, blocks) of a gzip member carrying the "SZ" block table (spzb200_gzip_table_info; no
    GPU).  CodecError(ERR_INVALID) for a member without one, or with one the parallel inflater would not trust."""
    buf = np.frombuffer(blob, np.uint8) if not isinstance(blob, np.ndarray) else np.ascontiguousarray(blob, np.uint8)
    size, blocks = C.c_uint64(0), C.c_int64(0)
    N.check(N.lib().spzb200_gzip_table_info(C.c_void_p(buf.ctypes.data if buf.size else None), buf.size, C.byref(size), C.byref(blocks)))
    return size.value, blocks.value


def shard_range(n: int, sh_degree: int, num_shards: int, index: int):
    """Contiguous point range of one shard (host logic, no GPU): spzb200_shard_range."""
    a, b = C.c_int64(0), C.c_int64(0)
    N.check(N.lib().spzb200_shard_range(n, sh_degree, num_shards, index, C.byref(a), C.byref(b)))
    return a.value, b.value


def tile_gaussians(sh_degree: int) -> int:
    return int(N.lib().spzb200_tile_gaussians(sh_degree))


def flip_bits(frm: int, to: int):
    p, q, s = C.c_uint32(0), C.c_uint32(0), C.c_uint32(0)
    N.lib().spzb200_flip_bits(frm, to, C.byref(p), C.byref(q), C.byref(s))
    return p.value, q.value, s.value


def build_tables():
    """The two host-built tables exactly as a context would build them (no GPU needed)."""
    thr, lut = np.zeros(256, np.float32), np.zeros(256, np.float32)
    N.check(N.lib().spzb200_build_tables(thr.ctypes.data_as(N._f32p), lut.ctypes.data_as(N._f32p)))
    return thr, lut


def ply_property_names(sh_degree: int):
    """Property order the reference's PLY writer emits (load-spz.cc:892-916)."""
    d = SH_DIM[sh_degree]
    return (["x", "y", "z", "nx", "ny", "nz", "f_dc_0", "f_dc_1", "f_dc_2"] + [f"f_rest_{i}" for i in range(3 * d)] +
            ["opacity", "scale_0", "scale_1", "scale_2", "rot_0", "rot_1", "rot_2", "rot_3"])


def ply_rows_struct(rows, n: int, names, sh_degree: int, on_device: Optional[bool]) -> N.PlyRows:
    """SpzB200PlyRows for row-major vertex records with the given property names (one float each)."""
    col = {name: i for i, name in enumerate(names)}
    width = len(names)
    s = N.PlyRows()
    s.num_points, s.width, s.sh_degree = n, width, sh_degree
    s.rows = _ptr(rows, "f4", n * width, on_device, "rows")
    s.col_pos[:] = [col["x"], col["y"], col["z"]]
    s.col_scale[:] = [col["scale_0"], col["scale_1"], col["scale_2"]]
    s.col_rot[:] = [col["rot_1"], col["rot_2"], col["rot_3"], col["rot_0"]]  # file is wxyz
    s.col_alpha = col["opacity"]
    s.col_color[:] = [col["f_dc_0"], col["f_dc_1"], col["f_dc_2"]]
    rest = [col[f"f_rest_{i}"] for i in range(3 * SH_DIM[sh_degree])]
    s.col_rest[:] = rest + [0] * (45 - len(rest))
    return s


class Context:
    """One caller at a time (own one per host thread, or lease one per call with pooled=True).  Raises
    CodecError(ERR_NO_DEVICE) when there is no B200: the codec has no CPU path."""

    def __init__(self, device: int = 0, pooled: bool = False):
        """pooled=True leases a context from the process-wide pool (spzb200_acquire) instead of
        creating one; close() hands it back."""
        self._h = C.c_void_p(None)
        self.device = device
        self.pooled = pooled
        N.check((N.lib().spzb200_acquire if pooled else N.lib().spzb200_create)(device, C.byref(self._h)))

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            (N.lib().spzb200_release if self.pooled else N.lib().spzb200_destroy)(self._h)
            self._h = C.c_void_p(None)

    __del__ = close

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    # ---- facts and knobs --------------------------------------------------------------------
    def info(self) -> dict:
        sm, pm, kl = C.c_int32(0), C.c_int32(0), C.c_int64(0)
        N.check(N.lib().spzb200_info(self._h, C.byref(sm), C.byref(pm), C.byref(kl)))
        return {"sm_count": sm.value, "pack_mode": "cvt.pack" if pm.value else "alu", "kernel_launches": kl.value}

    def tables(self):
        thr, lut = np.zeros(256, np.float32), np.zeros(256, np.float32)
        N.check(N.lib().spzb200_get_tables(self._h, thr.ctypes.data_as(N._f32p), lut.ctypes.data_as(N._f32p)))
        return thr, lut

    def set_force_generic(self, on: bool):
        N.lib().spzb200_set_force_generic(self._h, int(on))

    def set_pack_mode(self, cvt: bool):
        N.lib().spzb200_set_pack_mode(self._h, int(cvt))

    def set_chunk_points(self, points: int):
        N.lib().spzb200_set_chunk_points(self._h, int(points))

    def selfcheck_division(self, part: int, pairs_per_thread: int = 0, seed: int = 1):
        """(wrong, checked) of spzb200_selfcheck_division: the quotients of the rotation packer against the device's IEEE division."""
        wrong, checked = C.c_uint64(0), C.c_uint64(0)
        N.check(N.lib().spzb200_selfcheck_division(self._h, int(part), int(pairs_per_thread), int(seed), C.byref(wrong), C.byref(checked)))
        return int(wrong.value), int(checked.value)

    def set_host_staging(self, bounce: int = 1, copy_threads: int = 0):
        """bounce: 0 never, 1 auto (large calls), 2 always -- see spzb200_set_host_staging."""
        N.lib().spzb200_set_host_staging(self._h, int(bounce), int(copy_threads))

    # ---- device-resident ---------------------------------------------------------------------
    @staticmethod
    def _stream_handle(stream) -> int:
        if stream is None:
            import torch
            return torch.cuda.current_stream().cuda_stream
        return stream.cuda_stream if hasattr(stream, "cuda_stream") else int(stream)

    def encode_device(self, cloud: CloudPlanes, frm: int = 0, out: Optional[PackedPlanes] = None, stream=None, version: int = 3) -> PackedPlanes:
        """version=2 writes first-three rotations (3 bytes each; parity unpinned, see spzb200_encode_device_as)."""
        if out is None:
            out = alloc_packed(cloud.n, cloud.sh_degree, version, device=cloud.positions.device)
        out.antialiased = cloud.antialiased
        out.version = version
        cs, ps = _cloud_struct(cloud, True), _packed_struct(out, True)
        N.check(N.lib().spzb200_encode_device_as(self._h, C.byref(cs), int(frm), int(version), C.byref(ps), C.c_void_p(self._stream_handle(stream))))
        out.fractional_bits, out.version = ps.fractional_bits, ps.version
        return out

    def decode_device(self, packed: PackedPlanes, to: int = 0, out: Optional[CloudPlanes] = None, stream=None) -> CloudPlanes:
        if out is None:
            out = alloc_cloud(packed.n, packed.sh_degree, device=packed.positions.device)
        out.antialiased = packed.antialiased
        ps, cs = _packed_struct(packed, True), _cloud_struct(out, True)
        N.check(N.lib().spzb200_decode_device(self._h, C.byref(ps), int(to), C.byref(cs), C.c_void_p(self._stream_handle(stream))))
        return out

    def quantize_device(self, cloud: CloudPlanes, frm: int = 0, to: Optional[int] = None, version: int = 3,
                        out: Optional[CloudPlanes] = None, stream=None) -> CloudPlanes:
        """decode_device(encode_device(cloud, frm, version=version), to), bit for bit, in one kernel that writes no
        packed planes (spzb200_quantize_device): the cloud an .spz file of `cloud` gives back.  to=None means
        to=frm.  out=cloud runs in place; any other overlap between the planes of `out` and `cloud` is refused.
        Wrong plane sizes, an SH degree outside 0..3, a version other than 2 or 3 and overlaps raise
        CodecError(ERR_INVALID) and leave `out` untouched."""
        if to is None:
            to = frm
        if cloud.sh_degree not in SH_DIM:
            raise N.CodecError(N.ERR_INVALID, f"quantize_device: sh_degree {cloud.sh_degree} not in 0..3")
        if out is None:
            out = alloc_cloud(cloud.n, cloud.sh_degree, device=cloud.positions.device)
        try:
            cs, os_ = _cloud_struct(cloud, True), _cloud_struct(out, True)
        except (TypeError, ValueError) as e:
            raise N.CodecError(N.ERR_INVALID, f"quantize_device: {e}") from e
        N.check(N.lib().spzb200_quantize_device(self._h, C.byref(cs), int(frm), int(to), int(version), C.byref(os_),
                                                C.c_void_p(self._stream_handle(stream))))
        out.antialiased = cloud.antialiased
        return out

    # ---- .spz files of device-resident clouds (the deflate stage on the device) ------------------
    def _take_bytes(self, rc: int, out: C.c_void_p, size: C.c_size_t) -> bytes:
        N.check(rc)
        try:
            return C.string_at(out.value, size.value)
        finally:
            N.lib().spzb200_free(out)

    def gzip_device(self, data, stream=None) -> bytes:
        """A contiguous uint8 CUDA tensor -> one gzip member, deflated on the device (spzb200_gzip_device)."""
        ptr = _ptr(data, "u1", data.numel(), True, "data")
        out, size = C.c_void_p(None), C.c_size_t(0)
        rc = N.lib().spzb200_gzip_device(self._h, C.c_void_p(ptr), data.numel(), C.byref(out), C.byref(size),
                                         C.c_void_p(self._stream_handle(stream)))
        return self._take_bytes(rc, out, size)

    def gunzip_device(self, blob, out=None, stream=None):
        """A block-table gzip member in host memory -> (uint8 CUDA tensor of its inflated bytes, on_device), via
        spzb200_gunzip_device: the bytes spzb200_gunzip(threads > 1) returns; on_device is True when the device
        inflater produced them.  `out`, if given, is a contiguous uint8 CUDA tensor of at least the inflated
        size; the result is its leading slice.  Otherwise one is allocated from the table's size."""
        buf = np.frombuffer(blob, np.uint8) if not isinstance(blob, np.ndarray) else np.ascontiguousarray(blob, np.uint8)
        if out is None:
            import torch
            size, _ = gzip_table_info(buf)
            out = torch.empty(size, dtype=torch.uint8, device=f"cuda:{self.device}")
        ptr = _ptr(out, "u1", out.numel(), True, "out")
        got, on_device = C.c_size_t(0), C.c_int32(0)
        N.check(N.lib().spzb200_gunzip_device(self._h, C.c_void_p(buf.ctypes.data if buf.size else None), buf.size, C.c_void_p(ptr),
                                              out.numel(), C.byref(got), C.byref(on_device), C.c_void_p(self._stream_handle(stream))))
        return out[:got.value], bool(on_device.value)

    def save_spz_device(self, cloud: CloudPlanes, frm: int = 0, antialiased: bool = False, stream=None) -> bytes:
        """The .spz file of a device cloud (spzb200_save_spz_device): what saveSpz writes, inflated."""
        cs = _cloud_struct(cloud, True)
        out, size = C.c_void_p(None), C.c_size_t(0)
        rc = N.lib().spzb200_save_spz_device(self._h, C.byref(cs), int(frm), int(bool(antialiased)), C.byref(out), C.byref(size),
                                             C.c_void_p(self._stream_handle(stream)))
        return self._take_bytes(rc, out, size)

    def load_spz_device(self, blob, to: int = 0, device=None, out: Optional[CloudPlanes] = None, stream=None):
        """.spz bytes -> (CloudPlanes of CUDA tensors, antialiased) via spzb200_load_spz_device.  `out`, if
        given, must match the file's point count and SH degree (spz_info)."""
        buf = np.frombuffer(blob, np.uint8) if not isinstance(blob, np.ndarray) else np.ascontiguousarray(blob, np.uint8)
        if out is None:
            n, deg = spz_info(buf)
            out = alloc_cloud(n, deg, device=device if device is not None else f"cuda:{self.device}")
        cs = _cloud_struct(out, True)
        aa = C.c_int32(0)
        N.check(N.lib().spzb200_load_spz_device(self._h, C.c_void_p(buf.ctypes.data if buf.size else None), buf.size, int(to), C.byref(cs),
                                                C.byref(aa), C.c_void_p(self._stream_handle(stream))))
        out.antialiased = bool(aa.value)
        return out, out.antialiased

    # ---- batches of .spz files: one inflate or deflate launch per batch (DESIGN.md section 10c) -------
    @staticmethod
    def _host_blobs(blobs):
        bufs = [np.frombuffer(b, np.uint8) if not isinstance(b, np.ndarray) else np.ascontiguousarray(b, np.uint8) for b in blobs]
        ptrs = (C.c_void_p * max(len(bufs), 1))(*[b.ctypes.data for b in bufs])
        sizes = (C.c_size_t * max(len(bufs), 1))(*[b.size for b in bufs])
        return bufs, ptrs, sizes

    def _take_all(self, rc: int, outs, sizes, count: int):
        N.check(rc)
        try:
            return [C.string_at(outs[i], sizes[i]) for i in range(count)]
        finally:
            for i in range(count):
                N.lib().spzb200_free(C.c_void_p(outs[i]))

    @staticmethod
    def _batch_failed(what: str, status, count: int):
        failed = [i for i in range(count) if status[i] != N.OK]
        raise N.CodecError(N.ERR_INVALID, f"{what}: inputs {failed} failed ({N.last_error()})", failed)

    def gzip_device_batch(self, tensors, stream=None) -> list:
        """gzip_device of each contiguous uint8 CUDA tensor, every segment of the batch in one set of deflate
        launches (spzb200_gzip_device_batch).  Entry i equals gzip_device(tensors[i]) byte for byte."""
        k = len(tensors)
        ptrs = (C.c_void_p * max(k, 1))(*[_ptr(t, "u1", t.numel(), True, f"tensors[{i}]") or None for i, t in enumerate(tensors)])
        sizes = (C.c_size_t * max(k, 1))(*[t.numel() for t in tensors])
        outs, got = (C.c_void_p * max(k, 1))(), (C.c_size_t * max(k, 1))()
        rc = N.lib().spzb200_gzip_device_batch(self._h, ptrs, sizes, k, outs, got, C.c_void_p(self._stream_handle(stream)))
        return self._take_all(rc, outs, got, k)

    def save_spz_device_batch(self, clouds, frm: int = 0, antialiased=False, stream=None) -> list:
        """save_spz_device of each cloud (spzb200_save_spz_device_batch): one plane-move launch and one set of
        deflate launches for the batch.  antialiased: one flag for all, or one per cloud."""
        k = len(clouds)
        flags = list(antialiased) if isinstance(antialiased, (list, tuple)) else [antialiased] * k
        if len(flags) != k:
            raise N.CodecError(N.ERR_INVALID, f"save_spz_device_batch: {len(flags)} antialiased flags for {k} clouds")
        structs = (N.Cloud * max(k, 1))(*[_cloud_struct(c, True) for c in clouds])
        aa = (C.c_int32 * max(k, 1))(*[int(bool(f)) for f in flags])
        outs, got = (C.c_void_p * max(k, 1))(), (C.c_size_t * max(k, 1))()
        rc = N.lib().spzb200_save_spz_device_batch(self._h, structs, k, int(frm), aa, outs, got, C.c_void_p(self._stream_handle(stream)))
        return self._take_all(rc, outs, got, k)

    def gunzip_device_batch(self, blobs, outs=None, stream=None) -> list:
        """gunzip_device of each block-table gzip member (spzb200_gunzip_device_batch): every table block of the
        batch in one inflate launch -> [(uint8 CUDA tensor, on_device)].  `outs`, if given, holds one
        contiguous uint8 CUDA tensor per member.  Raises CodecError(ERR_INVALID) whose `failed` lists the
        members that failed; the others' outputs are complete then."""
        import torch
        bufs, ptrs, sizes = self._host_blobs(blobs)
        k = len(bufs)
        if outs is None:
            outs = []
            for b in bufs:
                try:
                    n = gzip_table_info(b)[0]
                except N.CodecError:
                    n = 0  # the call gives this member's verdict
                outs.append(torch.empty(n, dtype=torch.uint8, device=f"cuda:{self.device}"))
        dst = (C.c_void_p * max(k, 1))(*[_ptr(o, "u1", o.numel(), True, f"outs[{i}]") for i, o in enumerate(outs)])
        cap = (C.c_size_t * max(k, 1))(*[o.numel() for o in outs])
        got, on_dev, status = (C.c_size_t * max(k, 1))(), (C.c_int32 * max(k, 1))(), (C.c_int32 * max(k, 1))()
        rc = N.lib().spzb200_gunzip_device_batch(self._h, ptrs, sizes, k, dst, cap, got, on_dev, status,
                                                 C.c_void_p(self._stream_handle(stream)))
        if rc == N.ERR_INVALID and any(status[i] for i in range(k)):
            self._batch_failed("gunzip_device_batch", status, k)
        N.check(rc)
        return [(outs[i][:got[i]], bool(on_dev[i])) for i in range(k)]

    def load_spz_device_batch(self, blobs, to: int = 0, device=None, outs=None, stream=None) -> list:
        """load_spz_device of each .spz file (spzb200_load_spz_device_batch): the device-route files' table
        blocks in one inflate launch and their planes in one move launch -> [(CloudPlanes, antialiased)].
        `outs`, if given, holds one CloudPlanes per file sized by spz_info.  Raises CodecError(ERR_INVALID)
        whose message and `failed` list the files that failed; their outs are untouched, the others' complete."""
        bufs, ptrs, sizes = self._host_blobs(blobs)
        k = len(bufs)
        if outs is None:
            dev = device if device is not None else f"cuda:{self.device}"
            outs = []
            for b in bufs:
                try:
                    n, deg = spz_info(b)
                except N.CodecError:
                    n, deg = 0, 0  # the call gives this file's verdict
                outs.append(alloc_cloud(n, deg, device=dev))
        structs = (N.Cloud * max(k, 1))(*[_cloud_struct(o, True) for o in outs])
        aa, status = (C.c_int32 * max(k, 1))(), (C.c_int32 * max(k, 1))()
        rc = N.lib().spzb200_load_spz_device_batch(self._h, ptrs, sizes, k, int(to), structs, aa, status,
                                                   C.c_void_p(self._stream_handle(stream)))
        if rc in (N.OK, N.ERR_INVALID):
            for i, o in enumerate(outs):
                if status[i] == N.OK:
                    o.antialiased = bool(aa[i])
        if rc == N.ERR_INVALID and any(status[i] for i in range(k)):
            self._batch_failed("load_spz_device_batch", status, k)
        N.check(rc)
        return [(o, o.antialiased) for o in outs]

    # ---- fused PLY-rows encoder ---------------------------------------------------------------
    def encode_ply_device(self, rows, n: int, names, sh_degree: int, frm: int = 0, out: Optional[PackedPlanes] = None, stream=None):
        if out is None:
            out = alloc_packed(n, sh_degree, 3, device=rows.device)
        rs, ps = ply_rows_struct(rows, n, names, sh_degree, True), _packed_struct(out, True)
        N.check(N.lib().spzb200_encode_ply_device(self._h, C.byref(rs), int(frm), C.byref(ps), C.c_void_p(self._stream_handle(stream))))
        out.fractional_bits, out.version = ps.fractional_bits, ps.version
        return out

    def encode_ply_host(self, rows, n: int, names, sh_degree: int, frm: int = 0, out: Optional[PackedPlanes] = None):
        if out is None:
            out = alloc_packed(n, sh_degree, 3, numpy_arrays=True)
        rs, ps, tm = ply_rows_struct(rows, n, names, sh_degree, False), _packed_struct(out, False), N.Timings()
        N.check(N.lib().spzb200_encode_ply_host(self._h, C.byref(rs), int(frm), C.byref(ps), C.byref(tm)))
        out.fractional_bits, out.version = ps.fractional_bits, ps.version
        return out, tm.as_dict()

    def decode_ply_device(self, packed: PackedPlanes, names, to: int = 0, out=None, stream=None):
        """Packed planes -> row-major .ply records (one float per name); returns the rows tensor."""
        import torch
        if out is None:
            out = torch.empty(packed.n * len(names), dtype=torch.float32, device=packed.positions.device)
        ps, rs = _packed_struct(packed, True), ply_rows_struct(out, packed.n, names, packed.sh_degree, True)
        N.check(N.lib().spzb200_decode_ply_device(self._h, C.byref(ps), int(to), C.byref(rs), C.c_void_p(self._stream_handle(stream))))
        return out

    def decode_ply_host(self, packed: PackedPlanes, names, to: int = 0, out=None):
        if out is None:
            out = np.empty(packed.n * len(names), np.float32)
        ps, rs, tm = _packed_struct(packed, False), ply_rows_struct(out, packed.n, names, packed.sh_degree, False), N.Timings()
        N.check(N.lib().spzb200_decode_ply_host(self._h, C.byref(ps), int(to), C.byref(rs), C.byref(tm)))
        return out, tm.as_dict()

    # ---- host pointers (numpy arrays or CPU tensors, pinned for overlap) ----------------------
    def encode_host(self, cloud: CloudPlanes, frm: int = 0, out: Optional[PackedPlanes] = None, version: int = 3):
        if out is None:
            out = alloc_packed(cloud.n, cloud.sh_degree, version, numpy_arrays=True)
        out.antialiased = cloud.antialiased
        out.version = version
        cs, ps, tm = _cloud_struct(cloud, False), _packed_struct(out, False), N.Timings()
        N.check(N.lib().spzb200_encode_host_as(self._h, C.byref(cs), int(frm), int(version), C.byref(ps), C.byref(tm)))
        out.fractional_bits, out.version = ps.fractional_bits, ps.version
        return out, tm.as_dict()

    def decode_host(self, packed: PackedPlanes, to: int = 0, out: Optional[CloudPlanes] = None):
        if out is None:
            out = alloc_cloud(packed.n, packed.sh_degree, numpy_arrays=True)
        out.antialiased = packed.antialiased
        ps, cs, tm = _packed_struct(packed, False), _cloud_struct(out, False), N.Timings()
        N.check(N.lib().spzb200_decode_host(self._h, C.byref(ps), int(to), C.byref(cs), C.byref(tm)))
        return out, tm.as_dict()


    # ---- batched per-gaussian access: PackedGaussians::unpack(i, c), load-spz.cc:383-463 --------
    @staticmethod
    def _conv(converter):
        if converter is None:
            return None, None
        conv = np.ascontiguousarray(converter, np.float32).reshape(-1)
        if conv.size != 21:
            raise ValueError("converter must hold 21 floats: flipP[3], flipQ[3], flipSh[15]")
        return conv, conv.ctypes.data_as(N._f32p)

    def unpack_gather_host(self, packed: PackedPlanes, indices=None, converter=None, n: Optional[int] = None) -> np.ndarray:
        """[n, 59] float32 (UnpackedGaussian rows) of the gaussians `indices` (None: the first n) of HOST planes."""
        idx = None if indices is None else np.ascontiguousarray(indices, np.int64).reshape(-1)
        count = idx.size if idx is not None else (packed.n if n is None else int(n))
        out = np.empty((count, UNPACKED_FLOATS), np.float32)
        keep, cp = self._conv(converter)
        ps = _packed_struct(packed, False)
        N.check(N.lib().spzb200_unpack_gather_host(self._h, C.byref(ps), None if idx is None else C.c_void_p(idx.ctypes.data), count, cp,
                                                   C.c_void_p(out.ctypes.data)))
        return out

    def unpack_records_host(self, records, version: int, fractional_bits: int, converter=None) -> np.ndarray:
        """[n, 59] float32 from n 65-byte PackedGaussian records (what at() returns)."""
        rec = np.ascontiguousarray(records, np.uint8).reshape(-1, RECORD_BYTES)
        out = np.empty((rec.shape[0], UNPACKED_FLOATS), np.float32)
        keep, cp = self._conv(converter)
        N.check(N.lib().spzb200_unpack_records_host(self._h, C.c_void_p(rec.ctypes.data), rec.shape[0], int(version), int(fractional_bits), cp,
                                                    C.c_void_p(out.ctypes.data)))
        return out

    def unpack_gather_device(self, packed: PackedPlanes, indices=None, converter=None, n: Optional[int] = None, out=None, stream=None):
        """The same on DEVICE planes with a device index tensor (int64) or None; returns a [n, 59] float32 tensor."""
        import torch
        count = indices.numel() if indices is not None else (packed.n if n is None else int(n))
        if out is None:
            out = torch.empty((count, UNPACKED_FLOATS), dtype=torch.float32, device=packed.positions.device)
        if indices is not None and (indices.dtype != torch.int64 or not indices.is_contiguous()):
            raise TypeError("indices must be a contiguous int64 tensor")
        keep, cp = self._conv(converter)
        ps = _packed_struct(packed, True)
        N.check(N.lib().spzb200_unpack_gather_device(self._h, C.byref(ps), None if indices is None else C.c_void_p(indices.data_ptr()), count, cp,
                                                     C.c_void_p(out.data_ptr()), C.c_void_p(self._stream_handle(stream))))
        return out


_straight_through_fn = None


def _straight_through():
    """The autograd.Function behind quantize_straight_through, defined on first use (torch is imported lazily)."""
    global _straight_through_fn
    if _straight_through_fn is None:
        import torch

        class QuantizeStraightThrough(torch.autograd.Function):
            @staticmethod
            def forward(fctx, codec_ctx, n, sh_degree, antialiased, frm, version, *planes):
                cloud = CloudPlanes(n, sh_degree, *planes, antialiased=antialiased)
                out = codec_ctx.quantize_device(cloud, frm, frm, version)
                # an output plane carries a gradient only when its input plane asks for one
                fctx.mark_non_differentiable(*[o for o, p in zip(out.planes(), planes) if p is None or not p.requires_grad])
                return out.planes()

            @staticmethod
            def backward(fctx, *grads):
                return (None,) * 6 + tuple(g if need else None for need, g in zip(fctx.needs_input_grad[6:], grads))

        _straight_through_fn = QuantizeStraightThrough
    return _straight_through_fn


def quantize_straight_through(ctx: Context, cloud: CloudPlanes, frm: int = 0, version: int = 3) -> CloudPlanes:
    """ctx.quantize_device(cloud, frm, frm, version) as an autograd op with the straight-through estimator: the
    forward pass is the codec's round trip, and the backward pass hands each plane's incoming gradient to the
    matching input plane unchanged, as if the round trip were the identity.  No gradient flows through the
    quantizer's steps (their true derivative is zero almost everywhere); this is the usual way to fine-tune a
    cloud with the quantizer in the loop.  The output is in the input's frame (to = frm), so the identity is
    the right Jacobian for the flips too.  Returns new planes; `cloud` is not modified."""
    planes = _straight_through().apply(ctx, cloud.n, cloud.sh_degree, cloud.antialiased, int(frm), int(version), *cloud.planes())
    return CloudPlanes(cloud.n, cloud.sh_degree, *planes, antialiased=cloud.antialiased)


RECORD_BYTES = 65      # sizeof(PackedGaussian), load-spz.h:28-37
UNPACKED_FLOATS = 59   # UnpackedGaussian, load-spz.h:13-24


def gather_records(packed: PackedPlanes, indices) -> np.ndarray:
    """PackedGaussians::at(i) (load-spz.cc:431-459) for a list of indices on host numpy planes: [n, 65] uint8.
    A pure byte gather (SH de-interleaved per channel, padded with 128); no codec arithmetic."""
    idx = np.asarray(indices, np.int64)
    d = SH_DIM[packed.sh_degree]
    half = packed.version in (1, 4)
    pb, rb = (6 if half else 9), (4 if packed.version >= 3 else 3)
    rec = np.zeros((idx.size, RECORD_BYTES), np.uint8)
    rec[:, 0:pb] = np.asarray(packed.positions).reshape(-1, pb)[idx]
    rec[:, 9:9 + rb] = np.asarray(packed.rotations).reshape(-1, rb)[idx]
    rec[:, 13:16] = np.asarray(packed.scales).reshape(-1, 3)[idx]
    rec[:, 16:19] = np.asarray(packed.colors).reshape(-1, 3)[idx]
    rec[:, 19] = np.asarray(packed.alphas)[idx]
    rec[:, 20:65] = 128
    if d:
        sh = np.asarray(packed.sh).reshape(-1, d, 3)[idx]
        for ch in range(3):
            rec[:, 20 + 15 * ch:20 + 15 * ch + d] = sh[:, :, ch]
    return rec


def encode_host_multi(devices, cloud: CloudPlanes, frm: int = 0, out: Optional[PackedPlanes] = None):
    """Shards by contiguous point range over `devices` inside one process (no collective)."""
    if out is None:
        out = alloc_packed(cloud.n, cloud.sh_degree, 3, numpy_arrays=True)
    devs = (C.c_int32 * len(devices))(*devices)
    cs, ps, tm = _cloud_struct(cloud, False), _packed_struct(out, False), N.Timings()
    N.check(N.lib().spzb200_encode_host_multi(devs, len(devices), C.byref(cs), int(frm), C.byref(ps), C.byref(tm)))
    out.fractional_bits, out.version = ps.fractional_bits, ps.version
    return out, tm.as_dict()


def decode_host_multi(devices, packed: PackedPlanes, to: int = 0, out: Optional[CloudPlanes] = None):
    if out is None:
        out = alloc_cloud(packed.n, packed.sh_degree, numpy_arrays=True)
    devs = (C.c_int32 * len(devices))(*devices)
    ps, cs, tm = _packed_struct(packed, False), _cloud_struct(out, False), N.Timings()
    N.check(N.lib().spzb200_decode_host_multi(devs, len(devices), C.byref(ps), int(to), C.byref(cs), C.byref(tm)))
    return out, tm.as_dict()
