"""ctypes wrapper over oracle/_ref/libojph_oracle.so (the UNMODIFIED reference behind a C harness;
oracle/ref_harness.cpp).  Test infrastructure only."""
import ctypes as C
import os
import sys
import numpy as np

_ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PATH = os.path.join(_ROOT, "oracle", "_ref", "libojph_oracle.so")


class RParams(C.Structure):
    _fields_ = [
        ("width", C.c_uint32), ("height", C.c_uint32), ("off_x", C.c_uint32), ("off_y", C.c_uint32),
        ("tile_w", C.c_uint32), ("tile_h", C.c_uint32), ("tile_off_x", C.c_uint32), ("tile_off_y", C.c_uint32),
        ("num_comps", C.c_uint32), ("bit_depth", C.c_uint32 * 16), ("is_signed", C.c_uint32 * 16),
        ("dx", C.c_uint32 * 16), ("dy", C.c_uint32 * 16),
        ("num_decomps", C.c_uint32), ("block_w", C.c_uint32), ("block_h", C.c_uint32),
        ("num_precincts", C.c_uint32), ("precinct_w", C.c_uint32 * 33), ("precinct_h", C.c_uint32 * 33),
        ("reversible", C.c_uint32), ("color_transform", C.c_uint32), ("prog_order", C.c_uint32),
        ("qstep", C.c_float), ("qfactor", C.c_uint32), ("tlm", C.c_uint32), ("tilepart_div", C.c_uint32),
        ("planar", C.c_int32),
        ("coc_present", C.c_uint32 * 16), ("coc_reversible", C.c_uint32 * 16), ("coc_num_decomps", C.c_uint32 * 16),
        ("coc_block_w", C.c_uint32 * 16), ("coc_block_h", C.c_uint32 * 16),
        ("coc_num_precincts", C.c_uint32 * 16), ("coc_precinct_w", (C.c_uint32 * 33) * 16), ("coc_precinct_h", (C.c_uint32 * 33) * 16),
        ("nlt_all", C.c_uint32), ("nlt_comp", C.c_uint32 * 16), ("nlt_seq", C.c_uint32 * 16), ("profile", C.c_uint32),
        ("qcc_calls", C.c_uint32 * 16), ("qcc_qstep", C.c_float * 16), ("qcc_qstep_seq", C.c_uint32 * 16),
        ("qcc_qfactor", C.c_uint32 * 16), ("qcc_ctype", C.c_uint32 * 16), ("qcc_qfactor_seq", C.c_uint32 * 16),
    ]


class RInfo(C.Structure):
    _fields_ = [
        ("width", C.c_uint32), ("height", C.c_uint32), ("off_x", C.c_uint32), ("off_y", C.c_uint32),
        ("num_comps", C.c_uint32), ("bit_depth", C.c_uint32 * 16), ("is_signed", C.c_uint32 * 16),
        ("dx", C.c_uint32 * 16), ("dy", C.c_uint32 * 16), ("comp_w", C.c_uint32 * 16), ("comp_h", C.c_uint32 * 16),
        ("num_decomps", C.c_uint32), ("reversible", C.c_uint32), ("color_transform", C.c_uint32),
    ]


_lib = None


def available():
    return os.path.exists(PATH)


def active(lib=None):
    """where the tests' reference answers come from: this build of the reference when it was made (OJB_GOLDEN=record
    also stores what it answers), else the stored answers, replayed through `lib` (None: the product library) and
    checked against the reference's digests (tests/refgolden.py; OJB_GOLDEN=replay forces them)"""
    import refgolden
    mode = os.environ.get("OJB_GOLDEN", "")
    if available() and mode == "record":
        return refgolden.Recorder(lib)
    if available() and mode != "replay":
        return sys.modules[__name__]
    return refgolden.Golden(lib)


def lib():
    global _lib
    if _lib is None:
        _lib = C.CDLL(PATH)
        _lib.ojr_last_error.restype = C.c_char_p
        _lib.ojr_irv_K.restype = C.c_float
        _lib.ojr_irv_step.restype = C.c_float
    return _lib


def to_rparams(p):
    """copy an openjph_b200 Params (same field layout by construction) into RParams"""
    r = RParams()
    C.memmove(C.byref(r), C.byref(p), C.sizeof(RParams))
    return r


def _set_comments(L, comments):
    comments = comments or []
    keep = [c.encode("latin-1") if isinstance(c, str) else bytes(c) for c in comments]
    n = len(keep)
    data = (C.c_char_p * max(n, 1))(*keep)
    lens = (C.c_uint16 * max(n, 1))(*[len(k) for k in keep])
    text = (C.c_uint16 * max(n, 1))(*[1 if isinstance(c, str) else 0 for c in comments])
    L.ojr_set_comments(data, lens, text, C.c_uint32(n))


def encode(p, planes, comments=None):
    L = lib()
    _set_comments(L, comments)
    r = to_rparams(p)
    arrs = [np.ascontiguousarray(a, np.int32) for a in planes]
    ptrs = (C.c_void_p * len(arrs))(*[a.ctypes.data for a in arrs])
    cap = sum(a.size for a in arrs) * 5 + (1 << 20)
    out = np.zeros(cap, np.uint8)
    n = C.c_uint64()
    rc = L.ojr_encode(C.byref(r), ptrs, out.ctypes.data_as(C.c_void_p), C.c_uint64(cap), C.byref(n))
    if rc != 0:
        raise RuntimeError("reference encode failed: " + L.ojr_last_error().decode())
    return out[:n.value].tobytes()


def encode_into(p, planes_i32, out):
    """encode into a caller-owned (pre-touched) uint8 buffer: nothing is allocated inside the call, so a timed
    loop measures the reference and not page faults.  planes_i32: contiguous int32 arrays.  Returns the length."""
    L = lib()
    r = to_rparams(p)
    ptrs = (C.c_void_p * len(planes_i32))(*[a.ctypes.data for a in planes_i32])
    n = C.c_uint64()
    rc = L.ojr_encode(C.byref(r), ptrs, out.ctypes.data_as(C.c_void_p), C.c_uint64(out.size), C.byref(n))
    if rc != 0:
        raise RuntimeError("reference encode failed: " + L.ojr_last_error().decode())
    return int(n.value)


def decode_into(buf, length, planes_i32):
    """decode `length` bytes of the uint8 array `buf` into caller-owned int32 planes (see encode_into)"""
    L = lib()
    ptrs = (C.c_void_p * len(planes_i32))(*[a.ctypes.data for a in planes_i32])
    rc = L.ojr_decode(buf.ctypes.data_as(C.c_void_p), C.c_uint64(length), ptrs, 0)
    if rc != 0:
        raise RuntimeError("reference decode failed: " + L.ojr_last_error().decode())


def decode(j2c, resilient=False):
    L = lib()
    buf = np.frombuffer(j2c, np.uint8)
    info = RInfo()
    rc = L.ojr_read_info(buf.ctypes.data_as(C.c_void_p), C.c_uint64(buf.size), C.byref(info))
    if rc != 0:
        raise RuntimeError("reference read_headers failed: " + L.ojr_last_error().decode())
    planes = [np.zeros((info.comp_h[c], info.comp_w[c]), np.int32) for c in range(info.num_comps)]
    ptrs = (C.c_void_p * info.num_comps)(*[a.ctypes.data for a in planes])
    rc = L.ojr_decode(buf.ctypes.data_as(C.c_void_p), C.c_uint64(buf.size), ptrs, 1 if resilient else 0)
    if rc != 0:
        raise RuntimeError("reference decode failed: " + L.ojr_last_error().decode())
    return planes, info


def decode_restricted(j2c, skip_read, skip_recon, resilient=False):
    """codestream::restrict_input_resolution(skip_read, skip_recon) then decode"""
    L = lib()
    buf = np.frombuffer(j2c, np.uint8)
    info = RInfo()
    rc = L.ojr_decode_restricted(buf.ctypes.data_as(C.c_void_p), C.c_uint64(buf.size), None, 0,
                                 C.c_uint32(skip_read), C.c_uint32(skip_recon), C.byref(info))
    if rc != 0:
        raise RuntimeError("reference read_headers/restrict failed: " + L.ojr_last_error().decode())
    planes = [np.zeros((info.comp_h[c], info.comp_w[c]), np.int32) for c in range(info.num_comps)]
    ptrs = (C.c_void_p * info.num_comps)(*[a.ctypes.data for a in planes])
    rc = L.ojr_decode_restricted(buf.ctypes.data_as(C.c_void_p), C.c_uint64(buf.size), ptrs, 1 if resilient else 0,
                                 C.c_uint32(skip_read), C.c_uint32(skip_recon), None)
    if rc != 0:
        raise RuntimeError("reference decode failed: " + L.ojr_last_error().decode())
    return planes, info


def read_image(path, kind, w, h, nc, bit_depth, subsampling=None):
    """the apps' file readers (ppm_in: kind 0, yuv_in: kind 1) -> si32 component planes"""
    L = lib()
    sub = subsampling or [(1, 1)] * nc
    dims = [((w + dx - 1) // dx, (h + dy - 1) // dy) for dx, dy in sub]
    planes = [np.zeros((ch, cw), np.int32) for cw, ch in dims]
    ptrs = (C.c_void_p * nc)(*[a.ctypes.data for a in planes])
    dx = (C.c_uint32 * nc)(*[s[0] for s in sub])
    dy = (C.c_uint32 * nc)(*[s[1] for s in sub])
    rc = L.ojr_read_image(path.encode(), kind, C.c_uint32(w), C.c_uint32(h), C.c_uint32(nc), C.c_uint32(bit_depth), dx, dy, ptrs)
    if rc != 0:
        raise RuntimeError("reference image read failed: " + L.ojr_last_error().decode())
    return planes


def write_image(path, kind, bit_depth, planes):
    """the apps' file writers (ppm_out: kind 0, yuv_out: kind 1)"""
    L = lib()
    nc = len(planes)
    arrs = [np.ascontiguousarray(a, np.int32) for a in planes]
    ptrs = (C.c_void_p * nc)(*[a.ctypes.data for a in arrs])
    cw = (C.c_uint32 * nc)(*[a.shape[1] for a in arrs])
    ch = (C.c_uint32 * nc)(*[a.shape[0] for a in arrs])
    rc = L.ojr_write_image(path.encode(), kind, C.c_uint32(nc), C.c_uint32(bit_depth), cw, ch, ptrs)
    if rc != 0:
        raise RuntimeError("reference image write failed: " + L.ojr_last_error().decode())


def encode_block(block, missing_msbs, variant=0):
    """block: (h, w) uint32 sign-magnitude; returns bytes"""
    L = lib()
    h, w = block.shape
    stride = (w + 15) & ~15
    buf = np.zeros((h + 1, stride), np.uint32)
    buf[:h, :w] = block
    out = np.zeros(65536, np.uint8)
    n = C.c_uint32()
    rc = L.ojr_encode_block32(buf.ctypes.data_as(C.c_void_p), missing_msbs, w, h, stride,
                              out.ctypes.data_as(C.c_void_p), out.size, C.byref(n), variant)
    if rc != 0:
        raise RuntimeError("reference block encode failed")
    return out[:n.value].tobytes()


def decode_block(data, w, h, missing_msbs, num_passes, len1, len2, causal=False, variant=0):
    L = lib()
    stride = (w + 15) & ~15
    out = np.zeros((h + 2, stride), np.uint32)
    src = np.frombuffer(bytes(data) + b"\0" * 64, np.uint8).copy()
    rc = L.ojr_decode_block32(src.ctypes.data_as(C.c_void_p), out.ctypes.data_as(C.c_void_p), missing_msbs,
                              num_passes, len1, len2, w, h, stride, 1 if causal else 0, variant)
    return out[:h, :w].copy(), rc == 0
