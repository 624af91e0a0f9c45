"""ctypes binding of libjxlfront.so -- the C++ host front end (jxlatte_b200/frontend/, include/jxlfront.h).

`parse(data)` turns .jxl bytes into a `ParsedImage`: the headers as a dict and, per frame, the post-entropy arrays the
CUDA reconstruction takes (numpy views into memory owned by the parsed image).  This is the sequential half of the
decoder (entropy decoding, MA-tree walks, headers); it runs on the host in the reference too (north_star).
"""
import ctypes as C
import json
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.path.join(_HERE, "libjxlfront.so")
SRC_DIR = os.path.join(_HERE, "frontend")
CXX = "/usr/bin/g++"
CXXFLAGS = ["-std=c++17", "-O2", "-g", "-fPIC", "-shared", "-ffp-contract=off", "-fopenmp", "-Wall"]


class InvalidBitstreamError(IOError):
    """InvalidBitstreamException (J/io/InvalidBitstreamException.java)."""


def build(force=False):
    srcs = [os.path.join(SRC_DIR, f) for f in sorted(os.listdir(SRC_DIR))] + [os.path.join(_HERE, "..", "include", "jxlfront.h")]
    if not force and os.path.exists(SO_PATH) and all(os.path.getmtime(s) <= os.path.getmtime(SO_PATH) for s in srcs):
        return SO_PATH
    r = subprocess.run([CXX] + CXXFLAGS + ["-o", SO_PATH, os.path.join(SRC_DIR, "api.cpp")], capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("g++ failed building libjxlfront.so:\n" + r.stdout + r.stderr)
    return SO_PATH


_lib = None


def lib():
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(SO_PATH)
        L.jxlf_decode.argtypes = [C.c_void_p, C.c_uint64, C.c_int32, C.POINTER(C.c_void_p)]
        L.jxlf_decode.restype = C.c_int32
        L.jxlf_free.argtypes = [C.c_void_p]
        L.jxlf_free.restype = None
        L.jxlf_error.argtypes = [C.c_void_p]
        L.jxlf_error.restype = C.c_char_p
        L.jxlf_describe.argtypes = [C.c_void_p]
        L.jxlf_describe.restype = C.c_char_p
        L.jxlf_array.argtypes = [C.c_void_p, C.c_int32, C.c_char_p, C.c_int32, C.POINTER(C.c_void_p), C.POINTER(C.c_int64), C.POINTER(C.c_int32)]
        L.jxlf_array.restype = C.c_int32
        L.jxlf_set_threads.argtypes = [C.c_int32]
        L.jxlf_set_threads.restype = None
        _lib = L
    return _lib


FLAG_HOST_TRANSFORMS = 1     # also undo the frame-level modular transforms on the host (tests / cross-checks)
FLAG_HEADERS_ONLY = 2
FLAG_LF_ONLY = 4             # parse each frame up to its LF groups only (include/jxlfront.h JXLF_LF_ONLY)
_DTYPES = {0: np.int32, 1: np.float32, 2: np.uint8}


class ParsedImage:
    def __init__(self, data, flags=0, strict=True, threads=None):
        L = lib()
        if threads is not None:
            L.jxlf_set_threads(int(threads))        # this thread's OpenMP team size for the sections of each frame
        buf = (C.c_uint8 * len(data)).from_buffer_copy(data)
        h = C.c_void_p()
        self.status = L.jxlf_decode(buf, len(data), flags, C.byref(h))
        self._h = h
        self.error = L.jxlf_error(h).decode("utf-8", "replace")
        self.info = json.loads(L.jxlf_describe(h).decode("utf-8"))
        if strict and self.status != 0:
            msg = self.error
            self.close()
            if self.status == -2:
                raise InvalidBitstreamError(msg)
            if self.status == -3:
                raise NotImplementedError(msg)
            raise RuntimeError(msg)

    def close(self):
        if self._h:
            lib().jxlf_free(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def frames(self):
        return self.info["frames"]

    def array(self, frame, name, index=0, shape=None, copy=True):
        """One named array of a frame (see jxlf_array in include/jxlfront.h): a numpy copy, or with copy=False a read-only
        view into the parsed image's own memory (valid until close())."""
        p, n, dt = C.c_void_p(), C.c_int64(), C.c_int32()
        if lib().jxlf_array(self._h, frame, name.encode(), index, C.byref(p), C.byref(n), C.byref(dt)) != 0:
            raise KeyError("%s[%d] of frame %d" % (name, index, frame))
        dtype = np.dtype(_DTYPES[dt.value])
        if n.value == 0:
            a = np.zeros(0, dtype)
        else:
            a = np.frombuffer((C.c_char * (n.value * dtype.itemsize)).from_address(p.value), dtype=dtype)
            a = a.copy() if copy else a
        return a.reshape(shape) if shape is not None else a

    def vardct_state(self, frame, copy=True):
        """The dict jxlatte_b200.host.Reconstructor.reconstruct() takes, for a VarDCT frame.  copy=False hands out views
        into the parsed image (no 12 B/px memcpy); they die with close()."""
        f = self.frames[frame]
        H, W = f["padded_height"], f["padded_width"]
        sx, sy = f["shift_x"], f["shift_y"]
        st = {"width": W, "height": H}
        st["qcoeff"] = [self.array(frame, "qcoeff", c, (H >> sy[c], W >> sx[c]), copy) for c in range(3)]
        st["lf"] = [self.array(frame, "lf", c, ((H // 8) >> sy[c], (W // 8) >> sx[c]), copy) for c in range(3)]
        if copy and not any(sx) and not any(sy):
            st["qcoeff"] = np.stack(st["qcoeff"])
            st["lf"] = np.stack(st["lf"])
        for k, shp in (("dct_select", (H // 8, W // 8)), ("block_origin", (H // 8, W // 8)), ("hf_mul", (H // 8, W // 8)),
                       ("sharpness", (H // 8, W // 8)), ("x_from_y", ((H + 63) // 64, (W + 63) // 64)), ("b_from_y", ((H + 63) // 64, (W + 63) // 64))):
            st[k] = self.array(frame, k, 0, shp)
        return st

    def lf_quantised(self, frame):
        """The LF planes BEFORE LFCoefficients' arithmetic, for the device LF kernel (jxlb200_lf_dequant): (lf_quant int32 [3, H/8, W/8]
        in X, Y, B order, extraPrecision per LF group, scaledDequant[3], kX, kB, adaptive smoothing?), or None when the frame takes its LF
        from an LF frame or is chroma-subsampled (the front end's own planes are used then)."""
        f = self.frames[frame]
        if f["flags"] & 32 or any(f["shift_x"]) or any(f["shift_y"]):
            return None
        try:
            q, ep, sd, kx, kb, smooth = self.lf_state(frame)
        except Exception:
            return None
        return np.stack(q), ep, sd, kx, kb, smooth

    def lf_state(self, frame):
        """The quantised LF image of a VarDCT frame, chroma-subsampled or not: ([lf_quant int32 (hb >> sy[c], wb >> sx[c]) for X, Y, B],
        extraPrecision per LF group, scaledDequant[3], kX, kB, adaptive smoothing?).  hb, wb are the padded frame size in blocks."""
        f = self.frames[frame]
        hb, wb = f["padded_height"] // 8, f["padded_width"] // 8
        q = [self.array(frame, "lf_quant", c, (hb >> f["shift_y"][c], wb >> f["shift_x"][c])) for c in range(3)]
        ep = self.array(frame, "lf_extra_precision", 0)
        if ep.size != ((hb + 255) // 256) * ((wb + 255) // 256):
            raise InvalidBitstreamError("frame %d has no extraPrecision for every LF group" % frame)
        f32 = np.float32
        kx = f32(f["base_corr_x"]) + (f32(f["x_factor_lf"]) - f32(128.0)) / f32(f["color_factor"])     # LFCoefficients.java:81-82
        kb = f32(f["base_corr_b"]) + (f32(f["b_factor_lf"]) - f32(128.0)) / f32(f["color_factor"])
        return q, ep, [f32(v) for v in f["scaled_dequant"]], kx, kb, not bool(f["flags"] & 128)

    def modular_channels(self, frame):
        m = self.frames[frame]["modular"]
        return [self.array(frame, "modular", i, (c["h"], c["w"])) for i, c in enumerate(m["channels"])]


def parse(data, flags=0, strict=True, threads=None):
    """threads: OpenMP threads for the sections of each frame, for this and later parses on the calling thread (jxlf_set_threads);
    None leaves the thread's setting as it is."""
    return ParsedImage(data, flags, strict, threads)


def parse_file(path, flags=0, strict=True):
    with open(path, "rb") as f:
        return ParsedImage(f.read(), flags, strict)
