"""The reference's answers without the reference build.

Every call the tests make into the reference build (tests/refharness.py) is recorded once, with oracle/_ref present,
as a digest of what the reference returned.  Without the build the call is replayed: this project's own library
(the same one the test checks; the plain-C restatement for single code-blocks) computes the answer from the same
input and the answer is accepted only when its digest is the reference's.  Where this project's answer differs from
the reference's by design (9/7 rounding ties), the difference is stored as a small patch keyed by the digest of this
project's answer, so the reference's exact result is rebuilt and checked; any other difference fails the test.

  OJB_GOLDEN=record OJB_GOLDEN_DIR=<dir> python -m pytest tests ...   (with oracle/_ref) one shard per process
  python tests/refgolden.py merge <dir>...                           folds shards into golden/reference_calls.json.xz
"""
import base64
import ctypes as C
import hashlib
import io
import json
import lzma
import os
import re
import struct
import sys
import zlib
import numpy as np

PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_calls.json.xz")
_store = None


def _h(*parts, n=20):
    h = hashlib.sha256()
    for x in parts:
        if isinstance(x, np.ndarray):
            h.update(repr((x.dtype.str, x.shape)).encode())
            h.update(np.ascontiguousarray(x).tobytes())
        elif isinstance(x, (bytes, bytearray, memoryview)):
            h.update(b"%d:" % len(x))
            h.update(bytes(x))
        elif isinstance(x, C.Structure):
            h.update(C.string_at(C.addressof(x), C.sizeof(x)))
        elif isinstance(x, (list, tuple)):
            h.update(b"[%d:%s]" % (len(x), _h(*x).encode()))
        else:
            h.update(repr(x).encode())
        h.update(b"|")
    return h.hexdigest()[:n]


def _planes(planes):
    return [np.ascontiguousarray(a, np.int32) for a in planes]


def _comments(comments):
    return [("t", c) if isinstance(c, str) else ("b", bytes(c)) for c in (comments or [])]


# ---- results: digest, patch against this project's answer, rebuild -------------------------------------------------
def _digest(kind, r):
    if r is None:
        return "none"
    if kind == "bytes":
        return _h(r, n=16)
    if kind == "planes":
        return _h(_planes(r), n=16)
    return _h(np.ascontiguousarray(r[0], np.uint32), bool(r[1]), n=16)          # "block": (samples, ok)


def _npz(**arrays):
    b = io.BytesIO()
    np.savez(b, **arrays)
    return b.getvalue()


_PIECE = 8192


def _window(ours, i):
    """the part of this project's bytes that a piece starting at offset i of the reference's is compared with:
    it must fit zlib's 32 KB window together with the piece"""
    return ours[max(0, i - 12288):i + 20480]


def _make_patch(kind, ours, want):
    if kind == "bytes":
        if ours is None:
            return b"F" + want
        # piece by piece, each compressed with the same stretch of this project's bytes as the preset dictionary
        out = [b"Z"]
        for i in range(0, len(want), _PIECE):
            z = zlib.compressobj(9, zdict=_window(ours, i) or b"\0")
            d = z.compress(want[i:i + _PIECE]) + z.flush()
            out.append(struct.pack("<I", len(d)) + d)
        return b"".join(out)
    if kind == "planes":
        want = _planes(want)
        if ours is not None and [a.shape for a in ours] == [b.shape for b in want]:
            return b"D" + _npz(**{"c%d" % i: b.astype(np.int64) - a for i, (a, b) in enumerate(zip(_planes(ours), want))})
        return b"F" + _npz(**{"c%d" % i: b for i, b in enumerate(want)})
    return b"F" + _npz(a=np.asarray(want[0], np.uint32), ok=np.array(bool(want[1])))


def _apply_patch(kind, ours, patch):
    mode, body = patch[:1], patch[1:]
    if kind == "bytes":
        if mode == b"F":
            return body
        out, pos, i = [], 0, 0
        while pos < len(body):
            n = struct.unpack("<I", body[pos:pos + 4])[0]
            out.append(zlib.decompressobj(zdict=_window(ours, i) or b"\0").decompress(body[pos + 4:pos + 4 + n]))
            pos += 4 + n
            i += _PIECE
        return b"".join(out)
    z = np.load(io.BytesIO(body))
    if kind == "planes":
        n = len(z.files)
        if mode == b"F":
            return [z["c%d" % i] for i in range(n)]
        return [(a.astype(np.int64) + z["c%d" % i]).astype(np.int32) for i, a in enumerate(_planes(ours))]
    return z["a"], bool(z["ok"])


def _pack(b):
    return base64.b64encode(lzma.compress(b)).decode()


def _unpack(s):
    return lzma.decompress(base64.b64decode(s))


def store():
    global _store
    if _store is None:
        if not os.path.exists(PATH):
            raise RuntimeError("%s is missing and oracle/_ref was not built" % PATH)
        with lzma.open(PATH, "rt") as f:
            _store = json.load(f)
    return _store


# ---- the project's own answers ---------------------------------------------------------------------------------------
class _Ours:
    def __init__(self, lib):
        self.lib = lib

    def encode(self, p, planes, comments):
        import openjph_b200 as ob
        return ob.Encoder(p, ob.I32, lib=self.lib, comments=comments).encode(_planes(planes))

    def decode(self, j2c, resilient, skip=None):
        import openjph_b200 as ob
        return ob.Decoder(resilient=resilient, lib=self.lib).decode(bytes(j2c), skip=skip)

    def encode_block(self, block, missing_msbs):
        import oracleport
        return oracleport.encode_block(np.ascontiguousarray(block, np.uint32), missing_msbs)

    def decode_block(self, data, w, h, missing_msbs, num_passes, len1, len2, causal):
        import oracleport
        return oracleport.decode_block(data, w, h, missing_msbs, num_passes, len1, len2, causal)

    @staticmethod
    def read_image(path, kind, w, h, nc, bit_depth, sub):
        """the sample layouts of the files the tests write: .ppm/.pgm (0), .yuv (1), 10/16-bit RGB .dpx (2)"""
        data = open(path, "rb").read()
        wide = bit_depth > 8
        if kind == 0:
            body = data[re.match(rb"P[56]\s+\d+\s+\d+\s+\d+\s", data).end():]
            a = np.frombuffer(body, ">u2" if wide else np.uint8).reshape(h, w, nc)
            return [a[:, :, c].astype(np.int32) for c in range(nc)]
        if kind == 1:
            out, pos = [], 0
            for dx, dy in sub:
                cw, ch = (w + dx - 1) // dx, (h + dy - 1) // dy
                n = cw * ch * (2 if wide else 1)
                out.append(np.frombuffer(data[pos:pos + n], "<u2" if wide else np.uint8).reshape(ch, cw).astype(np.int32))
                pos += n
            return out
        big = data[:4] == b"SDPX"
        start = struct.unpack(">I" if big else "<I", data[4:8])[0]
        if bit_depth == 10:
            words = np.frombuffer(data[start:start + 4 * w * h], ">u4" if big else "<u4").reshape(h, w)
            return [((words >> s) & 0x3FF).astype(np.int32) for s in (22, 12, 2)]
        row = (3 * w + 1) & ~1
        a = np.frombuffer(data[start:start + 2 * row * h], ">u2" if big else "<u2").reshape(h, row)[:, :3 * w].reshape(h, w, 3)
        return [a[:, :, c].astype(np.int32) for c in range(3)]

    @staticmethod
    def write_image(kind, bit_depth, planes):
        wide = bit_depth > 8
        if kind == 0:
            h, w = planes[0].shape
            head = b"%s\n%d %d\n%d\n" % (b"P6" if len(planes) == 3 else b"P5", w, h, (1 << bit_depth) - 1)
            return head + np.stack(planes, -1).astype(">u2" if wide else np.uint8).tobytes()
        return b"".join(p.astype("<u2" if wide else np.uint8).tobytes() for p in planes)


def _try(fn):
    try:
        return fn()
    except Exception:
        return None


class _Calls:
    """the refharness API; subclasses decide where an answer comes from (`_call`)"""

    def __init__(self, lib):
        self.ours = _Ours(lib)

    def encode(self, p, planes, comments=None):
        key = _h("encode", p, _planes(planes), _comments(comments))
        return self._call(key, "bytes", lambda R: R.encode(p, planes, comments),
                          lambda: self.ours.encode(p, planes, comments))

    def decode(self, j2c, resilient=False):
        key = _h("decode", bytes(j2c), bool(resilient))
        return self._call(key, "planes", lambda R: R.decode(j2c, resilient), lambda: self.ours.decode(j2c, resilient), info=True)

    def decode_restricted(self, j2c, skip_read, skip_recon, resilient=False):
        key = _h("decode_restricted", bytes(j2c), int(skip_read), int(skip_recon), bool(resilient))
        return self._call(key, "planes", lambda R: R.decode_restricted(j2c, skip_read, skip_recon, resilient),
                          lambda: self.ours.decode(j2c, resilient, (skip_read, skip_recon)), info=True)

    def encode_block(self, block, missing_msbs, variant=0):
        key = _h("encode_block", np.ascontiguousarray(block, np.uint32), int(missing_msbs), int(variant))
        return self._call(key, "bytes", lambda R: R.encode_block(block, missing_msbs, variant),
                          lambda: self.ours.encode_block(block, missing_msbs))

    def decode_block(self, data, w, h, missing_msbs, num_passes, len1, len2, causal=False, variant=0):
        key = _h("decode_block", bytes(data), w, h, missing_msbs, num_passes, len1, len2, bool(causal), int(variant))
        return self._call(key, "block", lambda R: R.decode_block(data, w, h, missing_msbs, num_passes, len1, len2, causal, variant),
                          lambda: self.ours.decode_block(data, w, h, missing_msbs, num_passes, len1, len2, causal))

    def read_image(self, path, kind, w, h, nc, bit_depth, subsampling=None):
        sub = subsampling or [(1, 1)] * nc
        key = _h("read_image", open(path, "rb").read(), kind, w, h, nc, bit_depth, [tuple(s) for s in sub])
        return self._call(key, "planes", lambda R: R.read_image(path, kind, w, h, nc, bit_depth, subsampling),
                          lambda: self.ours.read_image(path, kind, w, h, nc, bit_depth, sub))

    def write_image(self, path, kind, bit_depth, planes):
        def live(R):
            R.write_image(path, kind, bit_depth, planes)
            return open(path, "rb").read()
        data = self._call(_h("write_image", kind, bit_depth, _planes(planes)), "bytes", live,
                          lambda: self.ours.write_image(kind, bit_depth, _planes(planes)))
        with open(path, "wb") as f:
            f.write(data)


class Golden(_Calls):
    """replays the stored answers (no reference build needed)"""

    def __init__(self, lib):
        super().__init__(lib)
        self._capture, self._code = False, 0
        self._lib = _ErrorHook(self)

    def lib(self):
        return self._lib

    def _call(self, key, kind, live, ours_fn, info=False):
        rec = store().get(key)
        if rec is None:
            raise LookupError("no stored reference answer for this call (%s); record it with the reference build, "
                              "see tests/refgolden.py" % key)
        if "err" in rec:
            text, code = rec["err"]
            if self._capture:
                self._code = code
            elif code:
                sys.stderr.write("ojph error 0x%08X: %s\n" % (code, text))
                sys.stderr.flush()
            raise RuntimeError("reference: " + text)
        ours = _try(ours_fn)
        d = _digest(kind, ours)
        if d == rec["sha"]:
            r = ours
        else:
            patch = rec.get("patch", {}).get(d)
            assert patch is not None, "this answer differs from the reference's (digest %s, want %s)" % (d, rec["sha"])
            r = _apply_patch(kind, ours, _unpack(patch))
            assert _digest(kind, r) == rec["sha"], "patched answer does not rebuild the reference's"
        if info:
            import refharness
            ri = refharness.RInfo()
            raw = bytes.fromhex(rec["info"])
            C.memmove(C.byref(ri), raw, len(raw))
            return r, ri
        return r


# the reference's line kernels the tests call directly -> the restatement's kernel (oracle/ojph_oracle.c) and its arguments;
# all take (source, destination, ..., count) over 4-byte samples
_LINE = {
    "ojr_rev_convert_nlt_type3": ("oj_rev_convert_nlt3", lambda a: (a[0], a[1], (_val(a[2]) - 1).bit_length(), a[3])),
    "ojr_irv_convert_to_float_nlt_type3": ("oj_irv_to_float_nlt3", lambda a: a),
    "ojr_irv_convert_to_integer_nlt_type3": ("oj_irv_to_int_nlt3", lambda a: a),
}


def _val(x):
    return x.value if hasattr(x, "value") else x


def _line_io(name, args):
    n = 4 * _val(args[-1])
    src, dst = (C.cast(a, C.c_void_p).value for a in args[:2])
    return _h(name, C.string_at(src, n), [_val(a) for a in args[2:]]), lambda: C.string_at(dst, n)


class _ErrorHook:
    """what the tests read from the reference library itself: its error code capture and line kernels"""

    def __init__(self, g):
        def capture(on):
            g._capture, g._code = bool(on), 0
        self.ojr_capture_errors = capture
        self.ojr_last_error_code = lambda: g._code

    def __getattr__(self, name):
        port_name, adapt = _LINE[name]

        def call(*args):
            import oracleport
            key, out = _line_io(name, args)
            rec = store().get(key)
            if rec is None:
                raise LookupError("no stored reference answer for this call (%s)" % key)
            getattr(oracleport.lib(), port_name)(*adapt(args))
            assert _h(out(), n=16) == rec["sha"], "the restatement's %s differs from the reference's %s" % (port_name, name)
        return call


class _RecordingLib:
    def __init__(self, L):
        self._L = L

    def __getattr__(self, name):
        fn = getattr(self._L, name)
        if name not in _LINE:
            return fn

        def call(*args):
            r = fn(*args)
            key, out = _line_io(name, args)
            _emit(key, {"sha": _h(out(), n=16)})
            return r
        return call


class Recorder(_Calls):
    """calls the reference build and appends what it answered to a shard of the golden store"""

    def __init__(self, lib):
        super().__init__(lib)
        import refharness
        self.R = refharness

    def lib(self):
        return _RecordingLib(self.R.lib())

    def _error(self, live):
        """the reference's error code and text, with its message capture on for the repeat"""
        L = self.R.lib()
        L.ojr_last_error_code.restype = C.c_uint32
        L.ojr_last_error_text.restype = C.c_char_p
        code = int(L.ojr_last_error_code())
        if code:
            return code, (L.ojr_last_error_text() or b"").decode(errors="replace")
        L.ojr_capture_errors(1)
        try:
            _try(lambda: live(self.R))
            return int(L.ojr_last_error_code()), (L.ojr_last_error_text() or b"").decode(errors="replace")
        finally:
            L.ojr_capture_errors(0)

    def _call(self, key, kind, live, ours_fn, info=False):
        try:
            r = live(self.R)
        except RuntimeError as e:
            code, text = self._error(live)
            _emit(key, {"err": [text or str(e), code]})
            raise
        res = r[0] if info else r
        rec = {"sha": _digest(kind, res)}
        if info:
            rec["info"] = C.string_at(C.addressof(r[1]), C.sizeof(r[1])).hex()
        ours = _try(ours_fn)
        d = _digest(kind, ours)
        if d != rec["sha"]:
            rec["patch"] = {d: _pack(_make_patch(kind, ours, res))}
        _emit(key, rec)
        return r


def _emit(key, rec):
    d = os.environ["OJB_GOLDEN_DIR"]
    os.makedirs(d, exist_ok=True)
    with open(os.path.join(d, "shard-%d.jsonl" % os.getpid()), "a") as f:
        f.write(json.dumps([key, rec]) + "\n")


def merge(dirs, path=PATH):
    out = {}
    if os.path.exists(path):
        with lzma.open(path, "rt") as f:
            out = json.load(f)
    for d in dirs:
        for name in sorted(os.listdir(d)):
            if not name.endswith(".jsonl"):
                continue
            for line in open(os.path.join(d, name)):
                key, rec = json.loads(line)
                old = out.setdefault(key, rec)
                if old is not rec:
                    assert old.get("sha") == rec.get("sha") and old.get("err") == rec.get("err"), key
                    old.setdefault("patch", {}).update(rec.get("patch", {}))
    with lzma.open(path, "wt", preset=9 | lzma.PRESET_EXTREME) as f:
        json.dump(out, f, sort_keys=True, separators=(",", ":"))
    return len(out)


if __name__ == "__main__":
    if len(sys.argv) > 2 and sys.argv[1] == "merge":
        print("%d reference answers in %s" % (merge(sys.argv[2:]), PATH))
    else:
        sys.exit(__doc__)
