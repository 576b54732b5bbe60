"""Thin ctypes binding of the C ABI in include/cdsgpu.h (libcdsgpu.so).

This is plumbing for tests and bench.py: every call goes straight to the shared library; there is no Python or CPU
implementation of anything behind it, and loading fails loudly when the library has not been built.
"""
import ctypes as C
import os
import weakref

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libcdsgpu.so")

CDS_OK = 0
CDS_ERR_BAD_ARG = 1
CDS_ERR_SIZE_MISMATCH = 2
CDS_ERR_NO_DEVICE = 3
CDS_ERR_CUDA = 4
CDS_ERR_OOM = 5
CDS_ERR_CAPACITY = 6
CDS_ERR_UNSUPPORTED = 7
CDS_MAX_RECTS = 8


class CdsError(RuntimeError):
    def __init__(self, status, message):
        super().__init__("libcdsgpu status %d: %s" % (status, message))
        self.status = status
        self.message = message


class CdsIllegalArgument(CdsError, ValueError):
    """CDS_ERR_BAD_ARG / CDS_ERR_SIZE_MISMATCH: where the Java reference throws IllegalArgumentException."""


class Rect(C.Structure):
    _fields_ = [("x0", C.c_int32), ("y0", C.c_int32), ("x1", C.c_int32), ("y1", C.c_int32)]


class PixParams(C.Structure):
    _fields_ = [("mask_threshold", C.c_int32), ("data_threshold", C.c_int32), ("z_tolerance", C.c_double),
                ("xy_shift", C.c_int32), ("mirror", C.c_int32), ("n_rects", C.c_int32), ("rects", Rect * CDS_MAX_RECTS)]


class SearchStats(C.Structure):
    _fields_ = [("kernel_launches", C.c_int64), ("match_kernel_launches", C.c_int64), ("match_kernel_ms", C.c_double),
                ("total_device_ms", C.c_double), ("comparisons", C.c_int64), ("h2d_bytes", C.c_int64), ("d2h_bytes", C.c_int64),
                ("match_kernel", C.c_int64), ("chunked", C.c_int64), ("host_inflate_fallbacks", C.c_int64)]


class TiffInfo(C.Structure):
    _fields_ = [("width", C.c_int32), ("height", C.c_int32), ("compression", C.c_int32), ("samples_per_pixel", C.c_int32),
                ("bits_per_sample", C.c_int32), ("photometric", C.c_int32), ("planar_config", C.c_int32), ("rows_per_strip", C.c_int32),
                ("n_strips", C.c_int32), ("big_endian", C.c_int32), ("data_bytes", C.c_int64), ("decodable", C.c_int32), ("pad", C.c_int32)]


class TargetGroupsC(C.Structure):
    """cds_target_groups: group keys of the targets of a best-matches search."""
    _fields_ = [("line", C.POINTER(C.c_int32)), ("sample", C.POINTER(C.c_int32)), ("line_hash", C.POINTER(C.c_int32)), ("n_lines", C.c_int32),
                ("sample_hash", C.POINTER(C.c_int32)), ("n_samples", C.c_int32)]


_lib = None
_vp = C.c_void_p
_u8p = C.POINTER(C.c_uint8)
_u16p = C.POINTER(C.c_uint16)
_u32p = C.POINTER(C.c_uint32)
_i32p = C.POINTER(C.c_int32)
_i64p = C.POINTER(C.c_int64)
_f32p = C.POINTER(C.c_float)
_f64p = C.POINTER(C.c_double)

class PngInfo(C.Structure):
    _fields_ = [("width", C.c_int32), ("height", C.c_int32), ("bit_depth", C.c_int32), ("color_type", C.c_int32), ("interlace", C.c_int32),
                ("decodable", C.c_int32), ("data_bytes", C.c_int64)]


class ZipEntry(C.Structure):
    _fields_ = [("name_offset", C.c_int64), ("name_len", C.c_int32), ("method", C.c_int32), ("data_offset", C.c_int64),
                ("compressed_size", C.c_int64), ("size", C.c_int64), ("crc32", C.c_uint32), ("is_directory", C.c_int32)]


# name -> (restype, argtypes); the single source of truth for the Python side of the ABI
SIGNATURES = {
    "cds_abi_version": (C.c_int32, []),
    "cds_ctx_create": (C.c_int32, [_i32p, C.c_int32, C.POINTER(_vp)]),
    "cds_ctx_destroy": (None, [_vp]),
    "cds_ctx_num_devices": (C.c_int32, [_vp]),
    "cds_last_error": (C.c_char_p, [_vp]),
    "cds_ctx_set_option": (C.c_int32, [_vp, C.c_char_p, C.c_int64]),
    "cds_host_alloc": (C.c_int32, [_vp, C.c_uint64, C.POINTER(_vp)]),
    "cds_host_free": (C.c_int32, [_vp, _vp]),
    "cds_library_create": (C.c_int32, [_vp, C.c_int32, C.c_int32, C.c_int64, C.POINTER(_vp)]),
    "cds_library_destroy": (None, [_vp]),
    "cds_library_add_rgb": (C.c_int32, [_vp, _vp, C.c_int64, _i64p]),
    "cds_library_generate_synthetic": (C.c_int32, [_vp, C.c_uint64, C.c_int64, C.c_int64, _i64p]),
    "cds_library_size": (C.c_int64, [_vp]),
    "cds_library_clear": (C.c_int32, [_vp]),
    "cds_maskset_create": (C.c_int32, [_vp, C.c_int32, C.c_int32, C.POINTER(PixParams), C.POINTER(_vp)]),
    "cds_maskset_destroy": (None, [_vp]),
    "cds_maskset_add_rgb": (C.c_int32, [_vp, _vp, C.c_int32, _i32p]),
    "cds_maskset_size": (C.c_int32, [_vp]),
    "cds_maskset_get_mask_sizes": (C.c_int32, [_vp, _i32p]),
    "cds_search_dense": (C.c_int32, [_vp, _vp, _vp, _i32p, _u8p]),
    "cds_search_topk": (C.c_int32, [_vp, _vp, _vp, C.c_int32, C.c_double, _i32p, _i64p, _u8p, _i32p]),
    "cds_search_stream_rgb": (C.c_int32, [_vp, _vp, _vp, C.c_int64, C.c_int32, C.c_double, _i32p, _i64p, _u8p, _i32p]),
    "cds_search_stream_matches_rgb": (C.c_int32, [_vp, _vp, _vp, C.c_int64, C.c_double, C.c_int64, _i32p, _i64p, _i32p, _u8p, _i64p]),
    "cds_search_matches": (C.c_int32, [_vp, _vp, _vp, C.c_double, C.c_int64, _i32p, _i64p, _i32p, _u8p, _i64p]),
    "cds_tiff_probe": (C.c_int32, [_vp, C.c_int64, C.POINTER(TiffInfo)]),
    "cds_tiff_encode_bound": (C.c_int64, [C.c_int32, C.c_int32, C.c_int32]),
    "cds_tiff_encode_rgb": (C.c_int32, [_vp, C.c_int32, C.c_int32, C.c_int32, C.c_int32, _vp, C.c_int64, _i64p]),
    "cds_tiff_decode_rgb": (C.c_int32, [_vp, _vp, _i64p, C.c_int64, C.c_int32, C.c_int32, _vp]),
    "cds_maskset_add_tiff": (C.c_int32, [_vp, _vp, _i64p, C.c_int32, _i32p]),
    "cds_library_add_tiff": (C.c_int32, [_vp, _vp, _i64p, C.c_int64, _i64p]),
    "cds_search_stream_tiff": (C.c_int32, [_vp, _vp, _vp, _i64p, C.c_int64, C.c_int32, C.c_double, _i32p, _i64p, _u8p, _i32p]),
    "cds_search_stream_matches_tiff": (C.c_int32, [_vp, _vp, _vp, _i64p, C.c_int64, C.c_double, C.c_int64, _i32p, _i64p, _i32p, _u8p, _i64p]),
    "cds_score_pair_rgb": (C.c_int32, [_vp, _vp, C.c_int32, _vp, C.c_int32, C.c_int32, _i32p, _f64p, _i32p]),
    "cds_shape_maskset_create": (C.c_int32, [_vp, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.POINTER(Rect), C.c_int32, _vp, C.POINTER(_vp)]),
    "cds_shape_maskset_destroy": (None, [_vp]),
    "cds_shape_maskset_add_rgb": (C.c_int32, [_vp, _vp, C.c_int32, _i64p, _i64p]),
    "cds_shape_maskset_size": (C.c_int32, [_vp]),
    "cds_shape_score_pairs": (C.c_int32, [_vp, _vp, _vp, _vp, _vp, _vp, C.c_int64, _i32p, _i64p, C.c_int64, _i64p, _i64p, _u8p]),
    "cds_shape_score_pairs_tiff": (C.c_int32, [_vp, _vp, _vp, _i64p, _vp, _vp, _vp, C.c_int64, _i32p, _i64p, C.c_int64, _i64p, _i64p, _u8p]),
    "cds_make_zgap": (C.c_int32, [_vp, _vp, C.c_int64, C.c_int32, C.c_int32, C.c_int32, C.c_double, C.POINTER(Rect), C.c_int32, _vp]),
    "cds_shape_score_2d": (C.c_int64, [C.c_int64, C.c_int64]),
    "cds_normalized_score": (C.c_double, [C.c_int32, C.c_int64, C.c_int64, C.c_int64]),
    "cds_normalize_scores": (C.c_int32, [_i32p, _i64p, _i64p, C.c_int64, _f32p]),
    "cds_select_best_matches": (C.c_int32, [_i32p, _i32p, _i32p, C.c_int64, _i32p, C.c_int32, _i32p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, _i64p, _i64p]),
    "cds_java_string_hash": (C.c_int32, [C.c_char_p]),
    "cds_search_best_matches": (C.c_int32, [_vp, _vp, _vp, C.POINTER(TargetGroupsC), C.c_double, C.c_int32, C.c_int32, C.c_int32, C.c_int64,
                                            _i32p, _i64p, _i32p, _u8p, _i64p]),
    "cds_search_stream_best_matches_tiff": (C.c_int32, [_vp, _vp, _vp, _i64p, C.c_int64, C.POINTER(TargetGroupsC), C.c_double, C.c_int32, C.c_int32,
                                                        C.c_int32, C.c_int64, _i32p, _i64p, _i32p, _u8p, _i64p]),
    "cds_search_stream_best_matches_rgb": (C.c_int32, [_vp, _vp, _vp, C.c_int64, C.POINTER(TargetGroupsC), C.c_double, C.c_int32, C.c_int32,
                                                       C.c_int32, C.c_int64, _i32p, _i64p, _i32p, _u8p, _i64p]),
    "cds_debug_select_best_matches_device": (C.c_int32, [_vp, _i32p, _i64p, _i32p, _u8p, C.c_int64, C.POINTER(TargetGroupsC), C.c_int32, C.c_int32,
                                                         C.c_int32, _i64p, _i64p]),
    "cds_synth_rgb": (C.c_int32, [_vp, C.c_int32, C.c_uint64, C.c_int64, C.c_int64, C.c_int32, C.c_int32, C.c_int32, _vp]),
    "cds_synth_gradient": (C.c_int32, [_vp, C.c_uint64, C.c_int64, C.c_int64, C.c_int32, C.c_int32, C.c_int32, _vp]),
    "cds_get_last_stats": (C.c_int32, [_vp, C.POINTER(SearchStats)]),
    "cds_debug_encode_colors": (C.c_int32, [_vp, _vp, C.c_int64, C.c_int32, _u32p]),
    "cds_debug_class_intervals": (C.c_int32, [C.c_double, C.c_int32, C.c_int32, _u32p, _u32p, _u32p, _u32p]),
    "cds_tiff_decode_rgb_host": (C.c_int32, [_vp, C.c_int64, C.c_int32, C.c_int32, _vp]),
    "cds_tiff_to_packbits": (C.c_int32, [_vp, C.c_int64, _vp, C.c_int64, _i64p]),
    "cds_png_probe": (C.c_int32, [_vp, C.c_int64, C.POINTER(PngInfo)]),
    "cds_png_decode_gray16": (C.c_int32, [_vp, _vp, _i64p, C.c_int64, C.c_int32, C.c_int32, _vp]),
    "cds_debug_inflate_host": (C.c_int32, [_vp, C.c_int64, _vp, C.c_int64, _i64p, _i32p]),
    "cds_png_encode_bound": (C.c_int64, [C.c_int32, C.c_int32]),
    "cds_png_encode_gray16": (C.c_int32, [_vp, C.c_int32, C.c_int32, C.c_int32, _vp, C.c_int64, _i64p]),
    "cds_zip_index": (C.c_int32, [_vp, C.c_int64, C.POINTER(ZipEntry), C.c_int64, _i64p]),
    "cds_zip_find": (C.c_int64, [_vp, C.POINTER(ZipEntry), C.c_int64, C.c_char_p]),
    "cds_zip_read": (C.c_int32, [_vp, C.c_int64, C.POINTER(ZipEntry), _vp, C.c_int64]),
    "cds_shape_score_pairs_files": (C.c_int32, [_vp, _vp, _vp, _i64p, _vp, _i64p, _vp, _vp, C.c_int64, _i32p, _i64p, C.c_int64, _i64p, _i64p, _u8p]),
    "cds_pairq_create": (C.c_int32, [_vp, _vp, C.c_int32, C.c_int32, C.c_int32, C.POINTER(_vp)]),
    "cds_pairq_destroy": (None, [_vp]),
    "cds_pairq_score": (C.c_int32, [_vp, C.c_int32, C.c_uint64, _vp, C.c_int32, C.c_int32, _i32p, _f64p, _i32p]),
    "cds_pairq_get_stats": (C.c_int32, [_vp, _i64p, _i64p, _i64p]),
    "cds_debug_pairq_drive": (C.c_int32, [_vp, _vp, C.c_int64, C.POINTER(C.c_uint64), _i32p, _i64p, C.c_int64, C.c_int32, _i32p, _u8p, _f64p]),
    "cds_debug_slice_numbers": (C.c_int32, [_vp, _vp, C.c_int64, _u16p]),
    "cds_debug_occupancy": (C.c_int32, [_vp, _vp, C.c_int64, C.c_int32, C.c_int32, C.c_int32, _vp]),
    "cds_debug_library_bands": (C.c_int32, [_vp, C.c_int32, C.c_int32, _u8p]),
    "cds_debug_cand_config": (C.c_int32, [C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, _i32p, _i32p, _i32p, _i64p]),
    "cds_debug_stream_plan": (C.c_int32, [C.c_int32, C.c_int64, C.c_int64, _vp, C.c_int64, C.c_int64, _vp, _vp, _vp, _vp]),
    "cds_debug_tiff_codes": (C.c_int32, [_vp, _vp, _i64p, C.c_int64, C.c_int32, C.c_int32, C.c_int32, C.c_int32, _u32p, _u32p]),
}


def lib():
    """Loads libcdsgpu.so.  Raises if it has not been built: there is no fallback of any kind."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError("libcdsgpu.so is missing (%s): run `python -m colormipsearch_b200.build`; "
                               "there is no CPU fallback" % LIB_PATH)
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)      # AttributeError here = the library does not export what the header declares
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def _check(status, ctx=None):
    if status == CDS_OK:
        return
    msg = lib().cds_last_error(ctx)
    msg = msg.decode("utf-8", "replace") if msg else ""
    if status in (CDS_ERR_BAD_ARG, CDS_ERR_SIZE_MISMATCH):
        raise CdsIllegalArgument(status, msg)
    raise CdsError(status, msg)


def _ptr(a):
    return None if a is None else a.ctypes.data_as(_vp)


def make_rects(rects):
    rects = np.asarray(rects if rects is not None else [], dtype=np.int32).reshape(-1, 4)
    arr = (Rect * max(len(rects), 1))()
    for i, r in enumerate(rects):
        arr[i] = Rect(int(r[0]), int(r[1]), int(r[2]), int(r[3]))
    return arr, len(rects)


class Context:
    def __init__(self, device_ids=None, n_dev=None):
        h = _vp()
        if device_ids is not None:
            ids = (C.c_int32 * len(device_ids))(*device_ids)
            st = lib().cds_ctx_create(ids, len(device_ids), C.byref(h))
        else:
            st = lib().cds_ctx_create(None, 1 if n_dev is None else int(n_dev), C.byref(h))
        _check(st, None)
        self.h = h
        self._children = weakref.WeakSet()

    def close(self):
        if getattr(self, "h", None):
            for child in list(self._children):      # libraries / mask sets die before their context
                child.close()
            lib().cds_ctx_destroy(self.h)
            self.h = None

    __del__ = close

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    @property
    def num_devices(self):
        return lib().cds_ctx_num_devices(self.h)

    MATCH_KERNELS = {"auto": 0, "cand": 1, "band": 2, "gather": 3}

    def set_option(self, name, value):
        _check(lib().cds_ctx_set_option(self.h, name.encode(), int(value)), self.h)

    def set_match_kernel(self, which):
        self.set_option("match_kernel", self.MATCH_KERNELS[which])

    def host_alloc(self, nbytes):
        """Pinned host buffer as a numpy uint8 array (freed with host_free)."""
        p = _vp()
        _check(lib().cds_host_alloc(self.h, int(nbytes), C.byref(p)), self.h)
        buf = (C.c_uint8 * int(nbytes)).from_address(p.value)
        arr = np.frombuffer(buf, dtype=np.uint8)
        return arr, p

    def host_free(self, p):
        _check(lib().cds_host_free(self.h, p), self.h)

    def last_stats(self):
        s = SearchStats()
        _check(lib().cds_get_last_stats(self.h, C.byref(s)), self.h)
        return {f[0]: getattr(s, f[0]) for f in SearchStats._fields_}

    def synth_rgb(self, kind, seed, first_index, n, W, H, on_device=True):
        out = np.empty((n, H, W, 3), np.uint8)
        _check(lib().cds_synth_rgb(self.h, int(kind), int(seed), int(first_index), int(n), W, H, int(on_device), _ptr(out)), self.h)
        return out

    def synth_gradient(self, seed, first_index, n, W, H, on_device=True):
        out = np.empty((n, H, W), np.uint16)
        _check(lib().cds_synth_gradient(self.h, int(seed), int(first_index), int(n), W, H, int(on_device), _ptr(out)), self.h)
        return out

    def debug_encode_colors(self, rgb, data_threshold):
        rgb = np.ascontiguousarray(rgb, dtype=np.uint8).reshape(-1, 3)
        out = np.empty(len(rgb), np.uint32)
        _check(lib().cds_debug_encode_colors(self.h, _ptr(rgb), len(rgb), int(data_threshold), out.ctypes.data_as(_u32p)), self.h)
        return out

    def debug_tiff_codes(self, files, W, H, data_threshold, fused):
        """-> (codes uint32[n][H][W], valid uint32[n][H][6][vp]) of the TIFF files through the fused or the two-kernel ingest path"""
        blob, offsets = pack_files(files)
        n = len(offsets) - 1
        vp = (((W + 31) // 32) + 3) // 4 * 4
        codes = np.zeros((n, H, W), np.uint32)
        valid = np.zeros((n, H, 6, vp), np.uint32)
        _check(lib().cds_debug_tiff_codes(self.h, _ptr(blob), offsets.ctypes.data_as(_i64p), n, W, H, int(data_threshold), int(bool(fused)),
                                          codes.ctypes.data_as(_u32p), valid.ctypes.data_as(_u32p)), self.h)
        return codes, valid

    def debug_occupancy(self, valid, W, H, xy_shift):
        """valid bits [n][H][6][vp] (uint32) -> occupancy tile rows [n][(H + 3) // 4][row pitch] (cds_debug_occupancy)."""
        valid = np.ascontiguousarray(valid, dtype=np.uint32)
        n = valid.shape[0]
        tp = ((W + 7) // 8 + 3) // 4 * 4
        nzw = ((6 * tp + 31) // 32 + 3) // 4 * 4
        out = np.empty((n, (H + 3) // 4, 7 * tp + nzw), np.uint32)
        _check(lib().cds_debug_occupancy(self.h, valid.ctypes.data_as(_vp), n, W, H, xy_shift, out.ctypes.data_as(_vp)), self.h)
        return out

    def debug_slice_numbers(self, rgb):
        rgb = np.ascontiguousarray(rgb, dtype=np.uint8).reshape(-1, 3)
        out = np.empty(len(rgb), np.uint16)
        _check(lib().cds_debug_slice_numbers(self.h, _ptr(rgb), len(rgb), out.ctypes.data_as(_u16p)), self.h)
        return out

    def make_zgap(self, rgb, threshold, radius, rects):
        rgb = np.ascontiguousarray(rgb, dtype=np.uint8)
        if rgb.ndim == 3:
            rgb = rgb[None]
        n, H, W, _ = rgb.shape
        out = np.empty_like(rgb)
        ra, nr = make_rects(rects)
        _check(lib().cds_make_zgap(self.h, _ptr(rgb), n, W, H, int(threshold), float(radius), ra, nr, _ptr(out)), self.h)
        return out


def synth_rgb_host(kind, seed, first_index, n, W, H):
    """Host build of the synthetic generator (no device needed)."""
    out = np.empty((n, H, W, 3), np.uint8)
    _check(lib().cds_synth_rgb(None, int(kind), int(seed), int(first_index), int(n), W, H, 0, _ptr(out)))
    return out


def synth_gradient_host(seed, first_index, n, W, H):
    out = np.empty((n, H, W), np.uint16)
    _check(lib().cds_synth_gradient(None, int(seed), int(first_index), int(n), W, H, 0, _ptr(out)))
    return out


class Library:
    def __init__(self, ctx, W, H, capacity):
        self.ctx = ctx
        self.W, self.H = W, H
        h = _vp()
        _check(lib().cds_library_create(ctx.h, W, H, int(capacity), C.byref(h)), ctx.h)
        self.h = h
        ctx._children.add(self)

    def close(self):
        if getattr(self, "h", None):
            lib().cds_library_destroy(self.h)
            self.h = None

    __del__ = close

    def add_rgb(self, rgb):
        rgb = np.ascontiguousarray(rgb, dtype=np.uint8)
        if rgb.ndim == 3:
            rgb = rgb[None]
        if rgb.shape[1:] != (self.H, self.W, 3):
            raise CdsIllegalArgument(CDS_ERR_SIZE_MISMATCH, "image shape %s does not match the library (%d, %d)" % (rgb.shape, self.H, self.W))
        first = C.c_int64()
        _check(lib().cds_library_add_rgb(self.h, _ptr(rgb), rgb.shape[0], C.byref(first)), self.ctx.h)
        return first.value

    def add_rgb_ptr(self, ptr, n):
        first = C.c_int64()
        _check(lib().cds_library_add_rgb(self.h, ptr, int(n), C.byref(first)), self.ctx.h)
        return first.value

    def add_tiff(self, files):
        """cds_library_add_tiff.  files: a list of bytes objects, or a (blob, offsets) pair (see pack_files)."""
        blob, offsets = pack_files(files)
        first = C.c_int64()
        _check(lib().cds_library_add_tiff(self.h, _ptr(blob), offsets.ctypes.data_as(_i64p), len(offsets) - 1, C.byref(first)), self.ctx.h)
        return first.value

    def generate_synthetic(self, seed, first_synth_index, n):
        first = C.c_int64()
        _check(lib().cds_library_generate_synthetic(self.h, int(seed), int(first_synth_index), int(n), C.byref(first)), self.ctx.h)
        return first.value

    def clear(self):
        _check(lib().cds_library_clear(self.h), self.ctx.h)

    def __len__(self):
        return lib().cds_library_size(self.h)

    def debug_bands(self, data_threshold, xy_shift):
        """The rank-band bytes of the resident occupancy for these search parameters, uint8 [n][(H + 3) // 4][6 * tp]
        (cds_debug_library_bands)."""
        tp = ((self.W + 7) // 8 + 3) // 4 * 4
        out = np.zeros((len(self), (self.H + 3) // 4, 6 * tp), np.uint8)
        _check(lib().cds_debug_library_bands(self.h, int(data_threshold), int(xy_shift), out.ctypes.data_as(_u8p)), self.ctx.h)
        return out


class MaskSet:
    def __init__(self, ctx, W, H, mask_threshold, data_threshold, z_tolerance, xy_shift, mirror, rects):
        self.ctx = ctx
        self.W, self.H = W, H
        p = PixParams()
        p.mask_threshold = int(mask_threshold)
        p.data_threshold = int(data_threshold)
        p.z_tolerance = float(z_tolerance)
        p.xy_shift = int(xy_shift)
        p.mirror = int(bool(mirror))
        rects = np.asarray(rects if rects is not None else [], dtype=np.int32).reshape(-1, 4)
        p.n_rects = len(rects)
        for i, r in enumerate(rects[:CDS_MAX_RECTS]):
            p.rects[i] = Rect(int(r[0]), int(r[1]), int(r[2]), int(r[3]))
        h = _vp()
        _check(lib().cds_maskset_create(ctx.h, W, H, C.byref(p), C.byref(h)), ctx.h)
        self.h = h
        ctx._children.add(self)

    def close(self):
        if getattr(self, "h", None):
            lib().cds_maskset_destroy(self.h)
            self.h = None

    __del__ = close

    def add_rgb(self, rgb):
        rgb = np.ascontiguousarray(rgb, dtype=np.uint8)
        if rgb.ndim == 3:
            rgb = rgb[None]
        if rgb.shape[1:] != (self.H, self.W, 3):
            raise CdsIllegalArgument(CDS_ERR_SIZE_MISMATCH, "mask shape %s does not match the mask set (%d, %d)" % (rgb.shape, self.H, self.W))
        sizes = np.zeros(rgb.shape[0], np.int32)
        _check(lib().cds_maskset_add_rgb(self.h, _ptr(rgb), rgb.shape[0], sizes.ctypes.data_as(_i32p)), self.ctx.h)
        return sizes

    def add_tiff(self, files, blob_ptr=None):
        """cds_maskset_add_tiff.  files: a list of bytes objects or a (blob, offsets) pair -> mask sizes."""
        blob, offsets = pack_files(files)
        n = len(offsets) - 1
        sizes = np.zeros(n, np.int32)
        ptr = blob_ptr if blob_ptr is not None else _ptr(blob)
        _check(lib().cds_maskset_add_tiff(self.h, ptr, offsets.ctypes.data_as(_i64p), n, sizes.ctypes.data_as(_i32p)), self.ctx.h)
        return sizes

    def add_rgb_ptr(self, ptr, n):
        sizes = np.zeros(n, np.int32)
        _check(lib().cds_maskset_add_rgb(self.h, ptr, int(n), sizes.ctypes.data_as(_i32p)), self.ctx.h)
        return sizes

    def __len__(self):
        return lib().cds_maskset_size(self.h)

    def sizes(self):
        out = np.zeros(max(len(self), 1), np.int32)
        _check(lib().cds_maskset_get_mask_sizes(self.h, out.ctypes.data_as(_i32p)), self.ctx.h)
        return out[: len(self)]

    def search_dense(self, library):
        M, T = len(self), len(library)
        scores = np.zeros((M, T), np.int32)
        mirrored = np.zeros((M, T), np.uint8)
        _check(lib().cds_search_dense(self.ctx.h, self.h, library.h, scores.ctypes.data_as(_i32p), mirrored.ctypes.data_as(_u8p)), self.ctx.h)
        return scores, mirrored

    def search_topk(self, library, k, pct_positive_pixels=0.0):
        M = len(self)
        score = np.zeros((M, k), np.int32)
        target = np.full((M, k), -1, np.int64)
        mirrored = np.zeros((M, k), np.uint8)
        count = np.zeros(M, np.int32)
        _check(lib().cds_search_topk(self.ctx.h, self.h, library.h, int(k), float(pct_positive_pixels),
                                     score.ctypes.data_as(_i32p), target.ctypes.data_as(_i64p),
                                     mirrored.ctypes.data_as(_u8p), count.ctypes.data_as(_i32p)), self.ctx.h)
        return score, target, mirrored, count

    def search_stream(self, targets_rgb, k, pct_positive_pixels=0.0, n=None):
        """cds_search_stream_rgb.  targets_rgb: a uint8 array [n][H][W][3], or a ctypes pointer together with n."""
        if n is None:
            targets_rgb = np.ascontiguousarray(targets_rgb, dtype=np.uint8)
            n = targets_rgb.shape[0] if targets_rgb.ndim == 4 else 1
            ptr = _ptr(targets_rgb)
        else:
            ptr = targets_rgb
        M = len(self)
        score = np.zeros((M, k), np.int32)
        target = np.full((M, k), -1, np.int64)
        mirrored = np.zeros((M, k), np.uint8)
        count = np.zeros(M, np.int32)
        _check(lib().cds_search_stream_rgb(self.ctx.h, self.h, ptr, int(n), int(k), float(pct_positive_pixels),
                                           score.ctypes.data_as(_i32p), target.ctypes.data_as(_i64p),
                                           mirrored.ctypes.data_as(_u8p), count.ctypes.data_as(_i32p)), self.ctx.h)
        return score, target, mirrored, count

    def search_stream_tiff(self, files, k, pct_positive_pixels=0.0, blob_ptr=None):
        """cds_search_stream_tiff.  files: a list of bytes objects or a (blob, offsets) pair; blob_ptr overrides the blob's address
        (e.g. a pinned copy of it)."""
        blob, offsets = pack_files(files)
        n = len(offsets) - 1
        M = len(self)
        score = np.zeros((M, k), np.int32)
        target = np.full((M, k), -1, np.int64)
        mirrored = np.zeros((M, k), np.uint8)
        count = np.zeros(M, np.int32)
        ptr = blob_ptr if blob_ptr is not None else _ptr(blob)
        _check(lib().cds_search_stream_tiff(self.ctx.h, self.h, ptr, offsets.ctypes.data_as(_i64p), int(n), int(k), float(pct_positive_pixels),
                                            score.ctypes.data_as(_i32p), target.ctypes.data_as(_i64p),
                                            mirrored.ctypes.data_as(_u8p), count.ctypes.data_as(_i32p)), self.ctx.h)
        return score, target, mirrored, count

    def search_stream_matches_tiff(self, files, pct_positive_pixels=0.0, capacity=None):
        """cds_search_stream_matches_tiff: every pair that passes isMatch, targets given as TIFF files."""
        blob, offsets = pack_files(files)
        n = len(offsets) - 1
        cap = int(capacity) if capacity is not None else max(1024, 4 * len(self))
        for _ in range(2):
            mask = np.zeros(cap, np.int32); target = np.zeros(cap, np.int64); score = np.zeros(cap, np.int32); mir = np.zeros(cap, np.uint8)
            count = C.c_int64(0)
            st = lib().cds_search_stream_matches_tiff(self.ctx.h, self.h, _ptr(blob), offsets.ctypes.data_as(_i64p), int(n),
                                                      float(pct_positive_pixels), cap, mask.ctypes.data_as(_i32p), target.ctypes.data_as(_i64p),
                                                      score.ctypes.data_as(_i32p), mir.ctypes.data_as(_u8p), C.byref(count))
            if st == CDS_ERR_CAPACITY and capacity is None:
                cap = int(count.value)
                continue
            _check(st, self.ctx.h)
            c = int(count.value)
            return mask[:c], target[:c], score[:c], mir[:c]
        _check(st, self.ctx.h)

    def search_stream_matches(self, targets_rgb, pct_positive_pixels=0.0, capacity=None):
        """cds_search_stream_matches_rgb: every pair that passes isMatch -> (mask, target, score, mirrored) arrays.  With
        capacity=None the call is retried once with the size the library reports."""
        targets_rgb = np.ascontiguousarray(targets_rgb, dtype=np.uint8)
        n = targets_rgb.shape[0] if targets_rgb.ndim == 4 else 1
        cap = int(capacity) if capacity is not None else max(1024, 4 * len(self))
        for _ in range(2):
            mask = np.zeros(cap, np.int32); target = np.zeros(cap, np.int64); score = np.zeros(cap, np.int32); mir = np.zeros(cap, np.uint8)
            count = C.c_int64(0)
            st = lib().cds_search_stream_matches_rgb(self.ctx.h, self.h, _ptr(targets_rgb), int(n), float(pct_positive_pixels), cap,
                                                     mask.ctypes.data_as(_i32p), target.ctypes.data_as(_i64p), score.ctypes.data_as(_i32p),
                                                     mir.ctypes.data_as(_u8p), C.byref(count))
            if st == CDS_ERR_CAPACITY and capacity is None:
                cap = int(count.value)
                continue
            _check(st, self.ctx.h)
            c = int(count.value)
            return mask[:c], target[:c], score[:c], mir[:c]
        _check(st, self.ctx.h)

    def search_matches(self, library, pct_positive_pixels=0.0, capacity=None):
        """cds_search_matches: every pair that passes isMatch over a resident library."""
        cap = int(capacity) if capacity is not None else max(1024, 4 * len(self))
        for _ in range(2):
            mask = np.zeros(cap, np.int32); target = np.zeros(cap, np.int64); score = np.zeros(cap, np.int32); mir = np.zeros(cap, np.uint8)
            count = C.c_int64(0)
            st = lib().cds_search_matches(self.ctx.h, self.h, library.h, float(pct_positive_pixels), cap, mask.ctypes.data_as(_i32p),
                                          target.ctypes.data_as(_i64p), score.ctypes.data_as(_i32p), mir.ctypes.data_as(_u8p), C.byref(count))
            if st == CDS_ERR_CAPACITY and capacity is None:
                cap = int(count.value)
                continue
            _check(st, self.ctx.h)
            c = int(count.value)
            return mask[:c], target[:c], score[:c], mir[:c]
        _check(st, self.ctx.h)

    def _best_matches(self, call, capacity):
        """Runs call(capacity, mask, target, score, mirrored, count) of a *_best_matches entry; with capacity=None it is retried once with
        the number of selected pairs the library reports."""
        cap = int(capacity) if capacity is not None else max(1024, 4 * len(self))
        for _ in range(2):
            mask = np.zeros(cap, np.int32); target = np.zeros(cap, np.int64); score = np.zeros(cap, np.int32); mir = np.zeros(cap, np.uint8)
            count = C.c_int64(0)
            st = call(cap, mask.ctypes.data_as(_i32p), target.ctypes.data_as(_i64p), score.ctypes.data_as(_i32p), mir.ctypes.data_as(_u8p),
                      C.byref(count))
            if st == CDS_ERR_CAPACITY and capacity is None and count.value > cap:
                cap = int(count.value)
                continue
            _check(st, self.ctx.h)
            c = int(count.value)
            return mask[:c], target[:c], score[:c], mir[:c]
        _check(st, self.ctx.h)

    def search_best_matches(self, library, groups, pct_positive_pixels, top_lines, top_samples, top_matches, capacity=None):
        """cds_search_best_matches: per mask, the pairs ColorMIPProcessUtils.selectBestMatches keeps, selected on the device ->
        (mask, target, score, mirrored) arrays.  groups: TargetGroups indexed by library index."""
        g = groups.struct()
        return self._best_matches(lambda cap, *out: lib().cds_search_best_matches(
            self.ctx.h, self.h, library.h, C.byref(g), float(pct_positive_pixels), int(top_lines), int(top_samples), int(top_matches), cap, *out), capacity)

    def search_stream_best_matches_tiff(self, files, groups, pct_positive_pixels, top_lines, top_samples, top_matches, capacity=None):
        """cds_search_stream_best_matches_tiff: the same over TIFF files in host memory (groups indexed by file)."""
        blob, offsets = pack_files(files)
        g = groups.struct()
        return self._best_matches(lambda cap, *out: lib().cds_search_stream_best_matches_tiff(
            self.ctx.h, self.h, _ptr(blob), offsets.ctypes.data_as(_i64p), len(offsets) - 1, C.byref(g), float(pct_positive_pixels),
            int(top_lines), int(top_samples), int(top_matches), cap, *out), capacity)

    def search_stream_best_matches_rgb(self, targets_rgb, groups, pct_positive_pixels, top_lines, top_samples, top_matches, capacity=None):
        """cds_search_stream_best_matches_rgb: the same over RGB images in host memory (groups indexed by image)."""
        targets_rgb = np.ascontiguousarray(targets_rgb, dtype=np.uint8)
        g = groups.struct()
        return self._best_matches(lambda cap, *out: lib().cds_search_stream_best_matches_rgb(
            self.ctx.h, self.h, _ptr(targets_rgb), int(targets_rgb.shape[0]), C.byref(g), float(pct_positive_pixels),
            int(top_lines), int(top_samples), int(top_matches), cap, *out), capacity)

    def score_pair(self, mask_index, target_rgb):
        target_rgb = np.ascontiguousarray(target_rgb, dtype=np.uint8)
        s = C.c_int32()
        r = C.c_double()
        m = C.c_int32()
        _check(lib().cds_score_pair_rgb(self.ctx.h, self.h, int(mask_index), _ptr(target_rgb), target_rgb.shape[1], target_rgb.shape[0],
                                        C.byref(s), C.byref(r), C.byref(m)), self.ctx.h)
        return s.value, r.value, bool(m.value)


class PairQueue:
    """cds_pairq_*: the reference's single-pair call (calculateMatchingScore) behind a micro-batching queue with a device-side
    target cache.  score() blocks and may be called from many threads."""

    def __init__(self, ctx, maskset, max_batch=64, max_wait_us=50, cache_targets=256):
        self.ctx, self.ms = ctx, maskset
        h = _vp()
        _check(lib().cds_pairq_create(ctx.h, maskset.h, int(max_batch), int(max_wait_us), int(cache_targets), C.byref(h)), ctx.h)
        self.h = h
        ctx._children.add(self)

    def close(self):
        if getattr(self, "h", None):
            lib().cds_pairq_destroy(self.h)
            self.h = None

    __del__ = close

    def score(self, mask_index, target_rgb, key=0):
        target_rgb = np.ascontiguousarray(target_rgb, dtype=np.uint8)
        s, r, m = C.c_int32(), C.c_double(), C.c_int32()
        _check(lib().cds_pairq_score(self.h, int(mask_index), int(key), _ptr(target_rgb), target_rgb.shape[1], target_rgb.shape[0],
                                     C.byref(s), C.byref(r), C.byref(m)), None)
        return s.value, r.value, bool(m.value)

    def stats(self):
        r, b, u = C.c_int64(), C.c_int64(), C.c_int64()
        _check(lib().cds_pairq_get_stats(self.h, C.byref(r), C.byref(b), C.byref(u)), None)
        return {"requests": r.value, "batches": b.value, "uploads": u.value}

    def drive(self, targets_rgb, keys, pair_mask, pair_target, n_threads):
        """n_threads native threads call cds_pairq_score over the pair list -> (scores, mirrored, seconds)"""
        targets_rgb = np.ascontiguousarray(targets_rgb, dtype=np.uint8)
        keys = None if keys is None else np.ascontiguousarray(keys, dtype=np.uint64)
        pair_mask = np.ascontiguousarray(pair_mask, dtype=np.int32)
        pair_target = np.ascontiguousarray(pair_target, dtype=np.int64)
        n = len(pair_mask)
        scores = np.zeros(n, np.int32)
        mir = np.zeros(n, np.uint8)
        secs = C.c_double()
        _check(lib().cds_debug_pairq_drive(self.h, _ptr(targets_rgb), targets_rgb.shape[0], None if keys is None else keys.ctypes.data_as(C.POINTER(C.c_uint64)),
                                           pair_mask.ctypes.data_as(_i32p), pair_target.ctypes.data_as(_i64p), n, int(n_threads),
                                           scores.ctypes.data_as(_i32p), mir.ctypes.data_as(_u8p), C.byref(secs)), None)
        return scores, mir.astype(bool), secs.value


class ShapeMaskSet:
    def __init__(self, ctx, W, H, query_threshold, mirror, rects, border=0, roi=None):
        self.ctx = ctx
        self.W, self.H = W, H
        ra, nr = make_rects(rects)
        if roi is not None:
            roi = np.ascontiguousarray(roi, dtype=np.uint8)
        self._roi = roi
        h = _vp()
        _check(lib().cds_shape_maskset_create(ctx.h, W, H, int(query_threshold), int(border), int(bool(mirror)), ra, nr, _ptr(roi), C.byref(h)), ctx.h)
        self.h = h
        ctx._children.add(self)

    def close(self):
        if getattr(self, "h", None):
            lib().cds_shape_maskset_destroy(self.h)
            self.h = None

    __del__ = close

    def add_rgb(self, rgb):
        rgb = np.ascontiguousarray(rgb, dtype=np.uint8)
        if rgb.ndim == 3:
            rgb = rgb[None]
        n = rgb.shape[0]
        qm = np.zeros(n, np.int64)
        he = np.zeros(n, np.int64)
        _check(lib().cds_shape_maskset_add_rgb(self.h, _ptr(rgb), n, qm.ctypes.data_as(_i64p), he.ctypes.data_as(_i64p)), self.ctx.h)
        return qm, he

    def add_rgb_ptr(self, ptr, n):
        """masks already laid out as uint8[n][H][W][3] at a raw host address (e.g. pinned memory from Context.host_alloc)"""
        qm = np.zeros(n, np.int64)
        he = np.zeros(n, np.int64)
        _check(lib().cds_shape_maskset_add_rgb(self.h, ptr, int(n), qm.ctypes.data_as(_i64p), he.ctypes.data_as(_i64p)), self.ctx.h)
        return qm, he

    def __len__(self):
        return lib().cds_shape_maskset_size(self.h)

    def score_pairs(self, target_rgb, gradient, zgap_rgb, pair_mask, pair_target, has_variants=None):
        target_rgb = np.ascontiguousarray(target_rgb, dtype=np.uint8)
        n_targets = target_rgb.shape[0]
        gradient = None if gradient is None else np.ascontiguousarray(gradient, dtype=np.uint16)
        zgap_rgb = None if zgap_rgb is None else np.ascontiguousarray(zgap_rgb, dtype=np.uint8)
        has_variants = None if has_variants is None else np.ascontiguousarray(has_variants, dtype=np.uint8)
        pair_mask = np.ascontiguousarray(pair_mask, dtype=np.int32)
        pair_target = np.ascontiguousarray(pair_target, dtype=np.int64)
        n = len(pair_mask)
        gap = np.zeros(n, np.int64)
        he = np.zeros(n, np.int64)
        mir = np.zeros(n, np.uint8)
        _check(lib().cds_shape_score_pairs(self.ctx.h, self.h, _ptr(target_rgb), _ptr(gradient), _ptr(zgap_rgb), _ptr(has_variants),
                                           n_targets, pair_mask.ctypes.data_as(_i32p), pair_target.ctypes.data_as(_i64p), n,
                                           gap.ctypes.data_as(_i64p), he.ctypes.data_as(_i64p), mir.ctypes.data_as(_u8p)), self.ctx.h)
        return gap, he, mir.astype(bool)

    def score_pairs_files(self, tiff_files, png_files, zgap_rgb, pair_mask, pair_target, has_variants=None):
        """cds_shape_score_pairs_files: targets as TIFF files, gradient images as PNG files"""
        tblob, toff = pack_files(tiff_files)
        pblob, poff = pack_files(png_files)
        n_targets = len(toff) - 1
        assert len(poff) - 1 == n_targets
        zgap_rgb = None if zgap_rgb is None else np.ascontiguousarray(zgap_rgb, dtype=np.uint8)
        has_variants = None if has_variants is None else np.ascontiguousarray(has_variants, dtype=np.uint8)
        pair_mask = np.ascontiguousarray(pair_mask, dtype=np.int32)
        pair_target = np.ascontiguousarray(pair_target, dtype=np.int64)
        n = len(pair_mask)
        gap = np.zeros(n, np.int64)
        he = np.zeros(n, np.int64)
        mir = np.zeros(n, np.uint8)
        _check(lib().cds_shape_score_pairs_files(self.ctx.h, self.h, _ptr(tblob), toff.ctypes.data_as(_i64p), _ptr(pblob), poff.ctypes.data_as(_i64p),
                                                 _ptr(zgap_rgb), _ptr(has_variants), n_targets, pair_mask.ctypes.data_as(_i32p),
                                                 pair_target.ctypes.data_as(_i64p), n, gap.ctypes.data_as(_i64p), he.ctypes.data_as(_i64p),
                                                 mir.ctypes.data_as(_u8p)), self.ctx.h)
        return gap, he, mir.astype(bool)

    def score_pairs_tiff(self, files, gradient, zgap_rgb, pair_mask, pair_target, has_variants=None, blob_ptr=None):
        """cds_shape_score_pairs_tiff: targets as TIFF files (a list of bytes objects or a (blob, offsets) pair)."""
        blob, offsets = pack_files(files)
        n_targets = len(offsets) - 1
        gradient = None if gradient is None else np.ascontiguousarray(gradient, dtype=np.uint16)
        zgap_rgb = None if zgap_rgb is None else np.ascontiguousarray(zgap_rgb, dtype=np.uint8)
        has_variants = None if has_variants is None else np.ascontiguousarray(has_variants, dtype=np.uint8)
        pair_mask = np.ascontiguousarray(pair_mask, dtype=np.int32)
        pair_target = np.ascontiguousarray(pair_target, dtype=np.int64)
        n = len(pair_mask)
        gap = np.zeros(n, np.int64)
        he = np.zeros(n, np.int64)
        mir = np.zeros(n, np.uint8)
        ptr = blob_ptr if blob_ptr is not None else _ptr(blob)
        _check(lib().cds_shape_score_pairs_tiff(self.ctx.h, self.h, ptr, offsets.ctypes.data_as(_i64p), _ptr(gradient), _ptr(zgap_rgb),
                                                _ptr(has_variants), n_targets, pair_mask.ctypes.data_as(_i32p),
                                                pair_target.ctypes.data_as(_i64p), n, gap.ctypes.data_as(_i64p), he.ctypes.data_as(_i64p),
                                                mir.ctypes.data_as(_u8p)), self.ctx.h)
        return gap, he, mir.astype(bool)


def shape_score_2d(gap, he):
    return lib().cds_shape_score_2d(int(gap), int(he))


def normalized_score(pix, shape, max_pix, max_shape):
    return lib().cds_normalized_score(int(pix), int(shape), int(max_pix), int(max_shape))


def normalize_scores(pixel_scores, gaps, high_exprs):
    pixel_scores = np.ascontiguousarray(pixel_scores, dtype=np.int32)
    gaps = np.ascontiguousarray(gaps, dtype=np.int64)
    high_exprs = np.ascontiguousarray(high_exprs, dtype=np.int64)
    out = np.zeros(len(pixel_scores), np.float32)
    _check(lib().cds_normalize_scores(pixel_scores.ctypes.data_as(_i32p), gaps.ctypes.data_as(_i64p), high_exprs.ctypes.data_as(_i64p),
                                      len(pixel_scores), out.ctypes.data_as(_f32p)))
    return out


def class_intervals(z_tolerance, sector, rank):
    lo1, len1, lo2, len2 = C.c_uint32(), C.c_uint32(), C.c_uint32(), C.c_uint32()
    _check(lib().cds_debug_class_intervals(float(z_tolerance), int(sector), int(rank), C.byref(lo1), C.byref(len1), C.byref(lo2), C.byref(len2)))
    return lo1.value, len1.value, lo2.value, len2.value


def pack_files(files):
    """A list of bytes-like objects -> (uint8 blob, int64 offsets[n + 1]), the layout the *_tiff calls take.  A (blob, offsets) pair
    passes through."""
    if isinstance(files, tuple) and len(files) == 2 and isinstance(files[1], np.ndarray):
        blob, offsets = files
        return blob, np.ascontiguousarray(offsets, dtype=np.int64)
    offsets = np.zeros(len(files) + 1, np.int64)
    for i, f in enumerate(files):
        offsets[i + 1] = offsets[i] + len(f)
    blob = np.frombuffer(b"".join(bytes(f) for f in files), dtype=np.uint8) if len(files) else np.zeros(0, np.uint8)
    if blob.size == 0:
        blob = np.zeros(1, np.uint8)
    return blob, offsets


def tiff_probe(data):
    """cds_tiff_probe -> dict of the TIFF's tags (host only)."""
    buf = np.frombuffer(bytes(data), dtype=np.uint8)
    info = TiffInfo()
    _check(lib().cds_tiff_probe(_ptr(buf) if buf.size else None, buf.size, C.byref(info)))
    return {k: getattr(info, k) for k, _ in TiffInfo._fields_ if k != "pad"}


def tiff_encode_rgb(rgb, rows_per_strip=8, compression=32773):
    """cds_tiff_encode_rgb -> bytes of a little-endian RGB TIFF (host only)."""
    rgb = np.ascontiguousarray(rgb, dtype=np.uint8)
    H, W = rgb.shape[:2]
    cap = lib().cds_tiff_encode_bound(W, H, rows_per_strip)
    out = np.empty(cap, np.uint8)
    n = C.c_int64(0)
    _check(lib().cds_tiff_encode_rgb(_ptr(rgb), W, H, rows_per_strip, compression, _ptr(out), cap, C.byref(n)))
    return out[:n.value].tobytes()


def tiff_decode_rgb(ctx, files, W, H):
    """cds_tiff_decode_rgb: decodes TIFF files on the device -> uint8 [n][H][W][3]."""
    blob, offsets = pack_files(files)
    n = len(offsets) - 1
    out = np.empty((n, H, W, 3), np.uint8)
    _check(lib().cds_tiff_decode_rgb(ctx.h, _ptr(blob), offsets.ctypes.data_as(_i64p), n, W, H, _ptr(out)), ctx.h)
    return out


def stream_plan(n_devices, n_targets, chunk, offsets=None, byte_cap=0xC0000000):
    """cds_debug_stream_plan: the chunk plan of the streaming searches, as arrays (device, first, count).  No device needed."""
    cap = int(n_targets) + 64
    dev = np.zeros(cap, np.int32); first = np.zeros(cap, np.int64); cnt = np.zeros(cap, np.int64)
    n = C.c_int64()
    off = None if offsets is None else np.ascontiguousarray(offsets, dtype=np.int64)
    _check(lib().cds_debug_stream_plan(int(n_devices), int(n_targets), int(chunk), None if off is None else off.ctypes.data_as(_vp), int(byte_cap), cap,
                                        dev.ctypes.data_as(_vp), first.ctypes.data_as(_vp), cnt.ctypes.data_as(_vp), C.byref(n)))
    return dev[:n.value], first[:n.value], cnt[:n.value]


def cand_config(W, H, xy_shift, palette_entries, wide=False):
    """cds_debug_cand_config: (warps, rows per band, stages, shared-memory bytes) of a candidate-kernel launch.  No device needed."""
    warps, rows, stages, smem = C.c_int32(), C.c_int32(), C.c_int32(), C.c_int64()
    _check(lib().cds_debug_cand_config(int(W), int(H), int(xy_shift), int(palette_entries), int(bool(wide)), C.byref(warps), C.byref(rows),
                                       C.byref(stages), C.byref(smem)))
    return warps.value, rows.value, stages.value, smem.value


def tiff_decode_rgb_host(data, W, H):
    """cds_tiff_decode_rgb_host: any supported TIFF (none / PackBits / LZW) decoded on the host -> uint8 [H][W][3]"""
    buf = np.frombuffer(bytes(data), np.uint8)
    out = np.empty((H, W, 3), np.uint8)
    _check(lib().cds_tiff_decode_rgb_host(_ptr(buf), len(buf), W, H, _ptr(out)))
    return out


def tiff_to_packbits(data):
    buf = np.frombuffer(bytes(data), np.uint8)
    info = tiff_probe(bytes(data))
    cap = lib().cds_tiff_encode_bound(info["width"], info["height"], 8)
    out = np.empty(cap, np.uint8)
    n = C.c_int64()
    _check(lib().cds_tiff_to_packbits(_ptr(buf), len(buf), _ptr(out), cap, C.byref(n)))
    return out[: n.value].tobytes()


def debug_inflate_host(data, capacity, misalign=0):
    """raw DEFLATE data through the device's decoder built for one lane -> (bytes produced so far, reason: 0 = inflated);
    the data starts `misalign` bytes behind an 8-byte boundary (the bit reader loads whole words from aligned data)"""
    buf = np.zeros(len(data) + misalign + 8, np.uint64).view(np.uint8)
    buf[misalign:misalign + len(data)] = np.frombuffer(bytes(data), np.uint8)
    out = np.empty(max(1, capacity), np.uint8)
    n = C.c_int64()
    why = C.c_int32()
    lib().cds_debug_inflate_host(C.c_void_p(buf.ctypes.data + misalign), len(data), _ptr(out), int(capacity), C.byref(n), C.byref(why))
    return out[: n.value].tobytes(), int(why.value)


def png_probe(data):
    buf = np.frombuffer(bytes(data), np.uint8)
    info = PngInfo()
    _check(lib().cds_png_probe(_ptr(buf), len(buf), C.byref(info)))
    return {f: getattr(info, f) for f, _ in PngInfo._fields_}


def png_encode_gray16(pixels, filter_mode=-1):
    pixels = np.ascontiguousarray(pixels, dtype=np.uint16)
    H, W = pixels.shape
    cap = lib().cds_png_encode_bound(W, H)
    out = np.empty(cap, np.uint8)
    n = C.c_int64()
    _check(lib().cds_png_encode_gray16(_ptr(pixels), W, H, int(filter_mode), _ptr(out), cap, C.byref(n)))
    return out[: n.value].tobytes()


def png_decode_gray16(ctx, files, W, H):
    """cds_png_decode_gray16: PNG files (inflate and filter reconstruction on the device) -> uint16 [n][H][W]"""
    blob, offsets = pack_files(files)
    n = len(offsets) - 1
    out = np.empty((n, H, W), np.uint16)
    _check(lib().cds_png_decode_gray16(ctx.h, _ptr(blob), offsets.ctypes.data_as(_i64p), n, W, H, _ptr(out)), ctx.h)
    return out


class ZipArchive:
    """cds_zip_index / cds_zip_find / cds_zip_read over an archive held in memory."""

    def __init__(self, data):
        self.buf = np.frombuffer(bytes(data), np.uint8)
        n = C.c_int64()
        _check(lib().cds_zip_index(_ptr(self.buf), len(self.buf), None, 0, C.byref(n)))
        self.entries = (ZipEntry * max(1, n.value))()
        _check(lib().cds_zip_index(_ptr(self.buf), len(self.buf), self.entries, n.value, C.byref(n)))
        self.n = n.value

    def names(self):
        return [bytes(self.buf[e.name_offset:e.name_offset + e.name_len]).decode() for e in self.entries[: self.n]]

    def find(self, name):
        return int(lib().cds_zip_find(_ptr(self.buf), self.entries, self.n, name.encode()))

    def read(self, index):
        e = self.entries[index]
        out = np.empty(max(1, e.size), np.uint8)
        _check(lib().cds_zip_read(_ptr(self.buf), len(self.buf), C.byref(e), _ptr(out), e.size))
        return out[: e.size].tobytes()

    def stored_span(self, index):
        """(offset, size) of a stored entry inside the archive: usable in place, no copy"""
        e = self.entries[index]
        return (int(e.data_offset), int(e.size)) if e.method == 0 else None


def java_string_hash(s):
    return int(lib().cds_java_string_hash(s.encode("ascii")))


def _group_ids(keys):
    """key strings -> (dense ids in first-appearance order, Java hashCode() per id); blank keys count as "UNKNOWN"."""
    table, out = {}, []
    for k in keys:
        k = k if k and k.strip() else "UNKNOWN"            # StringUtils.defaultIfBlank
        out.append(table.setdefault(k, len(table)))
    names = sorted(table, key=table.get)
    return np.asarray(out, np.int32), np.asarray([java_string_hash(nm) for nm in names], np.int32)


class TargetGroups:
    """The group keys of the targets of a best-matches search (cds_target_groups): lines[i] / samples[i] = published name / neuron id
    of target i, as strings; ids and hashes are derived the way select_best_matches derives them."""

    def __init__(self, lines, samples):
        self.line, self.line_hash = _group_ids(lines)
        self.sample, self.sample_hash = _group_ids(samples)
        if len(self.line) != len(self.sample):
            raise ValueError("lines and samples must name the same targets")

    def __len__(self):
        return len(self.line)

    def struct(self):
        """The C struct; it points into this object's arrays, so keep the object alive while the struct is used."""
        def p(a):
            return a.ctypes.data_as(_i32p) if len(a) else None
        return TargetGroupsC(p(self.line), p(self.sample), p(self.line_hash), len(self.line_hash), p(self.sample_hash), len(self.sample_hash))


def debug_select_best_matches_device(ctx, mask, target, score, mirrored, groups, top_lines, top_samples_per_line, top_matches_per_sample):
    """cds_debug_select_best_matches_device: the device selection alone over a list sorted by (mask, score desc, target asc);
    returns indices into the list in output order."""
    mask = np.ascontiguousarray(mask, np.int32); target = np.ascontiguousarray(target, np.int64); score = np.ascontiguousarray(score, np.int32)
    mirrored = None if mirrored is None else np.ascontiguousarray(mirrored, np.uint8)
    n = len(mask)
    sel = np.zeros(max(n, 1), np.int64)
    cnt = C.c_int64(0)
    g = groups.struct()
    _check(lib().cds_debug_select_best_matches_device(ctx.h, mask.ctypes.data_as(_i32p), target.ctypes.data_as(_i64p), score.ctypes.data_as(_i32p),
                                                      None if mirrored is None else mirrored.ctypes.data_as(_u8p), n, C.byref(g), int(top_lines),
                                                      int(top_samples_per_line), int(top_matches_per_sample), sel.ctypes.data_as(_i64p),
                                                      C.byref(cnt)), ctx.h)
    return sel[: cnt.value]


def select_best_matches(lines, samples, scores, top_lines, top_samples_per_line, top_matches_per_sample):
    """ColorMIPProcessUtils.selectBestMatches over one mask's matches.  lines / samples: sequences of key strings (ASCII);
    returns the indices of the kept matches in the reference's output order."""
    lid, lhash = _group_ids(lines)
    sid, shash = _group_ids(samples)
    sc = np.ascontiguousarray(scores, np.int32)
    n = len(sc)
    sel = np.zeros(max(n, 1), np.int64)
    cnt = C.c_int64(0)
    _check(lib().cds_select_best_matches(lid.ctypes.data_as(_i32p), sid.ctypes.data_as(_i32p), sc.ctypes.data_as(_i32p), n,
                                         lhash.ctypes.data_as(_i32p), len(lhash), shash.ctypes.data_as(_i32p), len(shash),
                                         int(top_lines), int(top_samples_per_line), int(top_matches_per_sample),
                                         sel.ctypes.data_as(_i64p), C.byref(cnt)))
    return sel[: cnt.value]
