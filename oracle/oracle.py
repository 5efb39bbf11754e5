"""oracle/oracle.py -- TEST INFRASTRUCTURE ONLY.

ctypes loaders for the two CPU checkers:

  load_restatement()   oracle/liboracle.so       the plain-C restatement (oracle/avif_oracle.c)
  load_reference()     oracle/_ref/libavifref.so the UNMODIFIED reference translation units compiled in place
                                                 (oracle/Makefile), or None when it has not been built
  load_recorded_reference()                      the restatement, held call by call to the compiled reference's
                                                 recorded results (tests/golden/reference_digests.npz)

Both expose the same Python surface (class CpuChecker) so a test can run either against the GPU library.
Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may import this module;
the product package never does.
"""
import ctypes as C
import hashlib
import os
import subprocess
import sys

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_HERE)
_PKG_PY = os.path.join(_ROOT, "avif-format_b200", "python")
if _PKG_PY not in sys.path:
    sys.path.insert(0, _PKG_PY)

from avifgpu import abi  # noqa: E402  (declarations only, loads no native code)


class OracleError(RuntimeError):
    def __init__(self, status, message):
        super().__init__(f"status {status}: {message}")
        self.status = status


def build(quiet=True):
    """Compile liboracle.so and, when /root/reference is present, _ref/libavifref.so."""
    out = subprocess.run(["make", "-C", _HERE, "all"], capture_output=True, text=True)
    if out.returncode != 0:
        raise RuntimeError("oracle build failed:\n" + out.stdout + out.stderr)
    if not quiet:
        print(out.stdout)


class CpuChecker:
    """Uniform Python surface over liboracle.so (prefix avif_oracle_) or libavifref.so (prefix avifref_)."""

    def __init__(self, path, prefix, kind):
        self.lib = C.CDLL(path)
        self.prefix = prefix
        self.kind = kind  # "port" (restatement) or "reference" (compiled reference TUs)
        self.path = path
        f = self._fn
        f("last_error", C.c_char_p, [])
        f("libm_version", C.c_char_p, [])
        f("transfer_f32", C.c_int, [C.c_int32, C.c_float, C.c_void_p, C.c_void_p, C.c_size_t])
        f("hlg_ootf", C.c_int, [C.c_void_p, C.c_size_t, C.c_int32, C.c_float, C.c_float])
        f("hlg_inverse_ootf", C.c_int, [C.c_void_p, C.c_size_t, C.c_int32, C.c_float, C.c_float])
        f("premultiply_u8", C.c_uint8, [C.c_uint8, C.c_uint8])
        f("premultiply_u16", C.c_uint16, [C.c_uint16, C.c_uint16, C.c_uint16])
        f("premultiply_f32", C.c_float, [C.c_float, C.c_float, C.c_float])
        f("unpremultiply_u8", C.c_uint8, [C.c_uint8, C.c_uint8])
        f("unpremultiply_u16", C.c_uint16, [C.c_uint16, C.c_uint16, C.c_uint16])
        f("unpremultiply_f32", C.c_float, [C.c_float, C.c_float, C.c_float])
        f("premultiply_table_u16", None, [C.c_uint16, C.c_int, C.c_void_p])
        f("premultiply_table_u8", None, [C.c_int, C.c_void_p])
        f("get_yuv_coefficients", C.c_int, [C.POINTER(abi.Nclx), C.c_void_p])
        f("get_hlg_luma_coefficients", C.c_int, [C.c_int32, C.c_void_p])
        f("build_yuv_tables", C.c_int, [C.POINTER(abi.Nclx), C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p])
        f("encode_image", C.c_int, [C.POINTER(abi.EncodeDesc), C.c_void_p, C.c_int64, C.POINTER(abi.Planes)])
        f("decode_image", C.c_int, [C.POINTER(abi.DecodeDesc), C.POINTER(abi.Planes), C.c_void_p, C.c_int64])
        f("encode_image_mt", C.c_int, [C.POINTER(abi.EncodeDesc), C.c_void_p, C.c_int64, C.POINTER(abi.Planes), C.c_int32])
        f("decode_image_mt", C.c_int, [C.POINTER(abi.DecodeDesc), C.POINTER(abi.Planes), C.c_void_p, C.c_int64, C.c_int32])
        if prefix == "avif_oracle_":
            f("build_depth_lut", C.c_int, [C.c_int32, C.c_int32, C.c_void_p])
            f("rgb_codes_to_ycbcr_mt", C.c_int, [C.POINTER(abi.EncodeDesc), C.c_void_p, C.c_int64, C.POINTER(abi.Planes), C.c_int32])

    def _fn(self, name, restype, argtypes):
        fn = getattr(self.lib, self.prefix + name)
        fn.restype = restype
        fn.argtypes = argtypes
        setattr(self, "_" + name, fn)

    def _check(self, status):
        if status != 0:
            raise OracleError(status, self._last_error().decode("utf-8", "replace"))

    # ---- scalars ----------------------------------------------------------------------------------------
    def libm_version(self):
        return self._libm_version().decode()

    def transfer(self, function, values, param=0.0):
        values = np.ascontiguousarray(values, dtype=np.float32)
        out = np.empty_like(values)
        self._check(self._transfer_f32(function, param, values.ctypes.data, out.ctypes.data, values.size))
        return out

    def hlg_ootf(self, rgb, primaries, gamma, peak):
        rgb = np.ascontiguousarray(rgb, dtype=np.float32).copy()
        self._check(self._hlg_ootf(rgb.ctypes.data, rgb.size // 3, primaries, gamma, peak))
        return rgb

    def hlg_inverse_ootf(self, rgb, primaries, gamma, peak):
        rgb = np.ascontiguousarray(rgb, dtype=np.float32).copy()
        self._check(self._hlg_inverse_ootf(rgb.ctypes.data, rgb.size // 3, primaries, gamma, peak))
        return rgb

    def premultiply_table(self, max_value, unpremultiply=False):
        if max_value == 255:
            out = np.empty((256, 256), np.uint8)
            self._premultiply_table_u8(int(unpremultiply), out.ctypes.data)
        else:
            out = np.empty((max_value + 1, max_value + 1), np.uint16)
            self._premultiply_table_u16(max_value, int(unpremultiply), out.ctypes.data)
        return out

    def premultiply_samples(self, values, alphas, max_value, unpremultiply=False):
        """The 16-bit (un)premultiply of each (value, alpha) pair, one call of the scalar function per pair."""
        fn = self._unpremultiply_u16 if unpremultiply else self._premultiply_u16
        return np.array([fn(v, a, max_value) for v, a in zip(np.asarray(values).tolist(), np.asarray(alphas).tolist())], np.uint16)

    def yuv_coefficients(self, nclx):
        out = np.zeros(3, np.float32)
        self._check(self._get_yuv_coefficients(C.byref(nclx) if nclx is not None else None, out.ctypes.data))
        return out

    def hlg_luma_coefficients(self, primaries):
        out = np.zeros(3, np.float32)
        self._check(self._get_hlg_luma_coefficients(primaries, out.ctypes.data))
        return out

    def yuv_tables(self, nclx, bit_depth, monochrome, has_alpha=True):
        n = 1 << bit_depth
        y = np.zeros(n, np.float32)
        uv = None if monochrome else np.zeros(n, np.float32)
        a = np.zeros(n, np.float32) if has_alpha else None
        self._check(self._build_yuv_tables(C.byref(nclx) if nclx is not None else None, bit_depth, int(monochrome),
                                           y.ctypes.data, uv.ctypes.data if uv is not None else None,
                                           a.ctypes.data if a is not None else None))
        return y, uv, a

    def depth_lut(self, host_depth, image_bit_depth):
        out = np.zeros(256 if host_depth == 8 else 32769, np.uint16)
        self._check(self._build_depth_lut(host_depth, image_bit_depth, out.ctypes.data))
        return out

    # ---- images -----------------------------------------------------------------------------------------
    def encode(self, desc, rows, threads=1, pad=0, planes=None):
        """rows: (H, W*channels) host array.  Returns the list of 4 plane arrays (None where absent)."""
        rows = np.ascontiguousarray(rows)
        assert rows.dtype == abi.host_dtype(desc.host_depth)
        assert rows.shape == (desc.height, desc.width * desc.host_channels), rows.shape
        if planes is None:
            planes = alloc_planes(abi.encode_plane_shapes(desc), abi.code_dtype(desc.image_bit_depth), pad)
        p = abi.planes_from_arrays(planes)
        status = self._encode_image_mt(C.byref(desc), rows.ctypes.data, rows.strides[0] if rows.size else 0,
                                       C.byref(p), threads)
        self._check(status)
        return planes

    def decode(self, desc, planes, threads=1):
        """planes: list of 4 arrays/None (2-D).  Returns the (H, W*channels) host array."""
        channels = abi.decode_host_channels(desc)
        rows = np.zeros((desc.height, desc.width * channels), abi.host_dtype(desc.host_depth))
        p = abi.planes_from_arrays(planes)
        status = self._decode_image_mt(C.byref(desc), C.byref(p), rows.ctypes.data, rows.strides[0] if rows.size else 0,
                                       threads)
        self._check(status)
        return rows

    def rgb_codes_to_ycbcr(self, desc, interleaved, pad=0, threads=1, planes=None):
        interleaved = np.ascontiguousarray(interleaved)
        if planes is None:
            planes = alloc_planes(abi.encode_plane_shapes(desc), abi.code_dtype(desc.image_bit_depth), pad)
        p = abi.planes_from_arrays(planes)
        self._check(self._rgb_codes_to_ycbcr_mt(C.byref(desc), interleaved.ctypes.data, interleaved.strides[0], C.byref(p),
                                                threads))
        return planes


def alloc_planes(shapes, dtype, pad=0, fill=0xCD):
    """Planes with `pad` extra samples of row padding (views into wider buffers), filled with a sentinel."""
    out = []
    for shape in shapes:
        if shape is None:
            out.append(None)
            continue
        rows, cols = shape
        backing = np.full((max(rows, 0), cols + pad), fill, dtype=dtype)
        out.append(backing[:, :cols])
    return out


_cache = {}


def load_restatement():
    if "port" not in _cache:
        path = os.path.join(_HERE, "liboracle.so")
        if not os.path.exists(path):
            build()
        _cache["port"] = CpuChecker(path, "avif_oracle_", "port")
    return _cache["port"]


def load_reference():
    """The compiled reference, or None if oracle/_ref/libavifref.so is absent and cannot be built here."""
    if "reference" not in _cache:
        path = os.path.join(_HERE, "_ref", "libavifref.so")
        if not os.path.exists(path) and os.path.exists("/root/reference/src/common/ColorTransfer.cpp"):
            build()
        _cache["reference"] = CpuChecker(path, "avifref_", "reference") if os.path.exists(path) else None
    return _cache["reference"]


def best_checker():
    """The compiled reference when available, else the restatement."""
    return load_reference() or load_restatement()


# ---- the compiled reference's results, recorded -----------------------------------------------------------------
#
# The reference's sources are not part of this repository, so oracle/_ref is only built where they are at hand.  Elsewhere
# the tests that compare with the reference use RecordedReference: the restatement, held call by call to the results the
# compiled reference returned for the same calls.  tests/golden/reference_digests.npz keeps those results as SHA-256
# digests (16 bytes of the digest of the call, 16 of the digest of its result), which keeps the comparison bit-exact
# over inputs far too large to store.  To record them, where oracle/_ref is built:
#
#   AVIFGPU_RECORD_REFERENCE=tests/golden/reference_digests.npz \
#       python -m pytest tests/test_oracle_vs_reference.py tests/test_forward_roundtrip.py -m "not gpu"

REFERENCE_DIGESTS = os.path.join(_ROOT, "tests", "golden", "reference_digests.npz")
_UNKEYED = ("threads", "pad")  # how the work is split and laid out in memory; the tests hold that neither changes a result


def _feed(h, value):
    """Hashes a value by content: arrays by dtype, shape and bytes, ctypes structures by their bytes."""
    if isinstance(value, (np.ndarray, np.generic)):
        value = np.asarray(value)
        h.update(f"array {value.dtype.str} {value.shape};".encode())
        h.update(np.ascontiguousarray(value).tobytes())
    elif isinstance(value, (list, tuple)):
        h.update(f"list {len(value)};".encode())
        for item in value:
            _feed(h, item)
    elif isinstance(value, C.Structure):
        h.update(f"{type(value).__name__};".encode() + bytes(value))
    elif isinstance(value, OracleError):
        h.update(f"error {value.status} {value};".encode())
    elif value is None or isinstance(value, (bool, int, float, str, bytes)):
        h.update(f"{type(value).__name__} {value!r};".encode())
    else:
        raise TypeError(f"no digest for {type(value).__name__}")


def _digest(*values):
    h = hashlib.sha256()
    for value in values:
        _feed(h, value)
    return h.digest()[:16]


def _call(checker, name, args, kwargs):
    """(call digest, result digest, result, error) of checker.<name>(*args, **kwargs); an OracleError is a result too."""
    keyed = sorted((k, v) for k, v in kwargs.items() if k not in _UNKEYED)
    key = _digest(name, list(args), [list(kv) for kv in keyed])
    try:
        result, error = getattr(checker, name)(*args, **kwargs), None
    except OracleError as raised:
        result, error = None, raised
    return key, _digest(error if error is not None else result), result, error


class ReferenceRecorder:
    """Wraps the compiled reference and records the digest of every call and of its result."""

    def __init__(self, reference):
        self._reference = reference
        self.digests = {}

    def __getattr__(self, name):
        if not callable(getattr(self._reference, name)):
            return getattr(self._reference, name)

        def call(*args, **kwargs):
            key, outcome, result, error = _call(self._reference, name, args, kwargs)
            if self.digests.setdefault(key, outcome) != outcome:
                raise AssertionError(f"{name}: the compiled reference returned two results for one call (threads or pad changed it)")
            if error is not None:
                raise error
            return result
        return call

    def save(self, path):
        keys = sorted(self.digests)
        np.savez_compressed(path, calls=np.frombuffer(b"".join(keys), np.uint8).reshape(-1, 16),
                            results=np.frombuffer(b"".join(self.digests[k] for k in keys), np.uint8).reshape(-1, 16),
                            libm=np.array(self._reference.libm_version()))


class RecordedReference:
    """The restatement in the reference's place: each call runs the restatement and fails unless its result is the one the
    compiled reference recorded for the same call.  A call the recording does not hold fails as well."""

    def __init__(self, port, calls, results):
        self._port = port
        self._results = dict(zip(calls, results))

    def __getattr__(self, name):
        if not callable(getattr(self._port, name)):
            return getattr(self._port, name)

        def call(*args, **kwargs):
            key, outcome, result, error = _call(self._port, name, args, kwargs)
            expected = self._results.get(key)
            if expected is None:
                raise AssertionError(f"{name}: no recorded reference result for this call (record again, see oracle.py)")
            if expected != outcome:
                raise AssertionError(f"{name}: the restatement's result differs from the compiled reference's recorded one"
                                     + (f" (the restatement raised: {error})" if error is not None else ""))
            if error is not None:
                raise error
            return result
        return call


def load_recorded_reference():
    """RecordedReference over tests/golden/reference_digests.npz, or None where this libm is not the one the results were
    recorded with (float results are only defined together with their libm)."""
    if "recorded" not in _cache:
        port = load_restatement()
        data = np.load(REFERENCE_DIGESTS)
        same_libm = str(data["libm"]) == port.libm_version()
        _cache["recorded"] = RecordedReference(port, [bytes(k) for k in data["calls"]], [bytes(r) for r in data["results"]]) \
            if same_libm else None
    return _cache["recorded"]
